#!/usr/bin/env python
"""bench.py -- image-text pairs/sec through the ViLBERT forward on B200, BASELINE.json's metric.

    python bench.py --gpus N --steps K --warmup W                       # configs[1]: batch 64 / GPU, VQA head, 36 x 30
    python bench.py --impl reference --gpus N --steps K --warmup W      # the reference's CPU PyTorch path (oracle port)
    python bench.py --workload multitask --gpus 8                       # configs[2]: B = 512 global, VQA / NLVR2 / RefCOCO thirds
    python bench.py --workload retrieval --gpus 8 --steps 1             # configs[3]: 1000 x 1000 caption-image score matrix
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR    # + the last timed step's outputs as DIR/<name>.npy

A "step" is one forward of one batch of `--batch` pairs per GPU (vqa, multitask: batches shard over ranks with no collective,
SURVEY.md 8e -> weak scaling) or one whole score matrix (retrieval: captions shard over ranks, ONE NCCL all-gather of the score
blocks on the compute stream -> strong scaling).  Rank 0 prints ONE JSON line.

value      : whole-job pairs/s with inputs resident in HBM (device-pointer C-ABI call, CUDA-event timed, max over ranks)
e2e        : the same through the host-buffer C-ABI call (pinned host inputs -> H2D -> forward -> D2H logits)
roofline   : tensor-pipe roofline of the dominant kernel family (the tcgen05 GEMMs, 97 % of the FLOPs)
alt        : the other 16-bit operand format measured in the same run (configs[1] names bf16; the engine's default is fp16 --
             same tcgen05 kind::f16 rate, 3 more significand bits), each with its measured max-abs-error vs the fp32 oracle
cpu_baseline: the fp32 PyTorch oracle (port of the reference's eager forward, all heads as the reference runs them) timed on
             this box's host cores, rank 0 at N=1 only, bounded sample
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "image-text pairs/sec (VQA head, 36 regions x 30 tok)"
UNIT = "pairs/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="vqa", choices=["vqa", "multitask", "retrieval"])
    p.add_argument("--batch", type=int, default=64, help="pairs per GPU per step (vqa, multitask); pairs per forward (retrieval)")
    p.add_argument("--n-tokens", type=int, default=30)
    p.add_argument("--n-regions", type=int, default=36)
    p.add_argument("--rotate", type=int, default=8, help="distinct resident input batches cycled through (L2 defeat)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-graph", action="store_true")
    p.add_argument("--pdl", choices=["default", "on", "off"], default="default",
                   help="programmatic dependent launch: engine default (every kernel), forced on, or off")
    p.add_argument("--all-heads", action="store_true", help="compute the seven task heads instead of VQA only")
    p.add_argument("--dtype", default="both", choices=["both", "fp16", "bf16", "fp32x"],
                   help="tensor-core operand format.  both (default): the configs[1] line in bf16 and the engine default fp16 "
                        "as `alt`; fp32x = fp32-parity mode (split operands, 3x the tensor work)")
    p.add_argument("--inflight", type=int, default=2,
                   help="batches in flight per GPU: steps alternate over this many CUDA streams / engine workspace slots")
    p.add_argument("--e2e-inflight", type=int, default=0,
                   help="workspace slots the host-buffer (e2e) loop submits into; 0 = --inflight + 1 (1 when --inflight is 1)")
    p.add_argument("--ops-table", default="", help="write the per-shape kernel time table (isolated graph replays) to this file")
    p.add_argument("--fused-ln", action="store_true", help="cluster-LayerNorm GEMM epilogue instead of GEMM + row LayerNorm")
    p.add_argument("--captions", type=int, default=1000, help="retrieval: captions (rows of the score matrix)")
    p.add_argument("--images", type=int, default=1000, help="retrieval: images (columns)")
    p.add_argument("--no-reuse", action="store_true", help="retrieval: full forward per pair instead of cached prefixes")
    p.add_argument("--dump-outputs", default="", metavar="DIR",
                   help="after the timed steps, write what the timed path returned in its last step (rank 0's share) as "
                        "DIR/<name>.npy, float32, at most 64 MB in all")
    a = p.parse_args()
    if a.dump_outputs and a.impl == "reference":
        p.error("--dump-outputs records the GPU path's outputs; --impl reference has none")
    return a


def env_rank():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return {"bf16_burst": d["bf16_tflops"], "bf16_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "hbm": d["hbm_gbs"], "src": "measured"}
    except Exception:
        return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "src": "fallback"}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each tensor of `arrays` (name -> tensor) as out_dir/<name>.npy in float32.  When they add up to more than
    DUMP_BYTES, every array keeps the same share of its rows, picked by torch.randperm seeded with 0: the rows depend on the shape
    alone, so two runs with the same arguments write the same rows."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu() for k, v in arrays.items()}
    total = sum(v.numel() * 4 for v in arrays.values())
    share = min(1.0, DUMP_BYTES / total) if total else 1.0
    for name, v in arrays.items():
        if share < 1.0:
            n = max(1, int(v.shape[0] * share))
            rows = torch.randperm(v.shape[0], generator=torch.Generator().manual_seed(0))[:n].sort().values
            v = v[rows]
        np.save(os.path.join(out_dir, name + ".npy"), v.numpy())


def named_outputs(out):
    """The engine's 10-tuple -> {output name: tensor} for the outputs the step computed (attention maps excluded)."""
    from vilbert_b200 import _lib as L
    return {k: v for k, v in zip(L.OUTPUT_FIELDS, out[:9]) if v is not None}


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz, self.err = index, False, [], set(), None, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                     "hw_power_brake": 0x80, "sw_power_cap": 0x4, "sync_boost": 0x10}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
                time.sleep(0.003)
        except Exception as e:          # NVML missing: report it, never fail the bench
            self.err = repr(e)

    def result(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "error": self.err}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ reference arm
def oracle_model(sd, cfg_dict, num_labels):
    """The ONLY place bench.py touches oracle/: the CPU baseline legs and the in-run parity numbers."""
    import torch
    from oracle import vilbert_ref as R
    m = R.VILBertForVLTasks(R.RefConfig(**{k: v for k, v in cfg_dict.items() if k in R.DEFAULT_CONFIG}), num_labels=num_labels)
    m.load_state_dict(sd, strict=True)
    return m.eval()


CPU_THREADS = min(16, os.cpu_count() or 1)   # measured on the 128-vCPU GPU box: 8 -> 56, 16 -> 78, 32 -> 44, 64 -> 23, 128 -> 0.2 pairs/s


def time_oracle(model, req, steps, warmup, all_heads=True):
    import torch
    torch.set_num_threads(CPU_THREADS)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            model(*req, output_all_attention_masks=True, compute_pretraining_heads=all_heads)   # as the reference runs it
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    return times


def run_reference(args):
    rank, _, world = env_rank()
    if rank != 0:
        return
    import torch
    import vilbert_b200 as vb
    from vilbert_b200 import synthetic as S
    cfg = vb.BertConfig(task_specific_tokens=True, visualization=True)
    sd = S.synthetic_state_dict(cfg, seed=42)
    model = oracle_model(sd, cfg.to_dict(), 3129)
    # bounded sample: ~2400 pairs in total (about two minutes of host work), never more than the real batch
    ref_batch = max(4, min(args.batch, 2400 // max(1, args.steps)))
    req = S.synthetic_request(ref_batch, args.n_tokens, args.n_regions, seed=1234)
    steps = args.steps
    times = time_oracle(model, req, steps, max(1, min(args.warmup, 2)))
    total = sum(times)
    value = ref_batch * len(times) / total
    cores = CPU_THREADS
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"batch={args.batch} VQA forward, {args.n_regions} regions x {args.n_tokens} tokens "
                                   "(BASELINE.json configs[1]); reference arm = fp32 PyTorch oracle port on host cores, "
                                   "all heads + pre-training heads as the reference executes them",
                       "global_batch": args.batch, "parallelism": "cpu"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{len(times)} forwards of {ref_batch} pairs each (bounded sample of the batch-{args.batch} "
                                       f"workload; torch fp32, {torch.get_num_threads()} threads)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ B200 arm: shared pieces
def make_engine(args, sd, cfg, dtype, local_rank):
    import vilbert_b200 as vb
    return vb.VILBertForVLTasks.from_pretrained(sd, config=cfg, num_labels=3129, use_cuda_graph=not args.no_graph,
                                                use_pdl={"default": None, "on": True, "off": False}[args.pdl],
                                                compute_dtype=dtype, fused_layernorm=args.fused_ln).eval().cuda(local_rank)


def all_rank_ms(ms, world, dev):
    """-> (max over ranks, per-rank list)."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return ms, [ms]
    t = torch.tensor([ms], device=dev)
    out = torch.empty(world, device=dev)
    dist.all_gather_into_tensor(out, t)
    lst = [float(x) for x in out.tolist()]
    return max(lst), lst


def timed_loop(step, n_steps, warmup, streams, dev, world, sampler=None):
    """W warm-up steps, then exactly n_steps between barrier + synchronize on both sides, CUDA events; ms on this rank."""
    import torch
    import torch.distributed as dist
    nfl = len(streams)

    def fork():
        if nfl > 1:
            ev = torch.cuda.Event()
            ev.record()
            for s_ in streams:
                s_.wait_event(ev)

    def join():
        if nfl > 1:
            for s_ in streams:
                ev = torch.cuda.Event()
                ev.record(s_)
                torch.cuda.current_stream(dev).wait_event(ev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    out = None
    fork()
    for i in range(max(warmup, 3) * nfl):
        out = step(i)
    join()
    sync_all()
    if sampler is not None:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fork()
    for i in range(n_steps):
        out = step(i)
    join()
    e1.record()
    sync_all()
    if sampler is not None:
        sampler.stop_flag = True
    return e0.elapsed_time(e1), out, sync_all


def parity_rows(model, oracle, req, rows, select_idx=0):
    """max |engine - fp32 oracle| over `rows` of the batch (the engine's rows do not depend on their batch neighbours)."""
    import torch
    dev = torch.device("cuda", model._device)
    sub = [t[rows] for t in req]
    with torch.no_grad():
        torch.set_num_threads(CPU_THREADS)
        ref = oracle(*sub, compute_pretraining_heads=False)[select_idx]
    out = model(*[t.to(dev) for t in sub])[select_idx].cpu()
    return float((out - ref).abs().max()), float(ref.std())


# ------------------------------------------------------------------------------------------------ configs[1]: VQA
def measure_vqa(args, model, reqs, dev, world, rank, local_rank, select, with_profile):
    import torch
    from vilbert_b200 import _lib as L
    B, Tin, V = args.batch, args.n_tokens, args.n_regions
    n_launch, flops = model.plan_info(B, Tin, V, select)
    dreqs = [[t.to(dev) for t in r] for r in reqs]
    in_bytes = sum(t.numel() * t.element_size() for i, t in enumerate(reqs[0]) if i != 6)
    nfl = max(1, args.inflight if not args.no_graph else 1)
    streams = [torch.cuda.Stream(device=dev) for _ in range(nfl)] if nfl > 1 else [torch.cuda.current_stream(dev)]

    def step(i):
        # step i = one forward of one batch; consecutive steps go to alternating streams / workspace slots so that the
        # kernels of one batch fill SMs the other leaves idle (every step still runs start to finish inside the timed region)
        if nfl == 1:
            return model(*dreqs[i % args.rotate], select=select)
        with torch.cuda.stream(streams[i % nfl]):
            return model(*dreqs[i % args.rotate], select=select, slot=i % nfl)

    sampler = ClockSampler(local_rank)
    ms_local, out, sync_all = timed_loop(step, args.steps, args.warmup, streams, dev, world, sampler)
    ms, per_rank = all_rank_ms(ms_local, world, dev)
    sampler.join(timeout=1.0)
    assert torch.isfinite(out[0]).all(), "non-finite logits"
    value = B * world * args.steps / (ms * 1e-3)

    # ---- e2e: host-buffer C-ABI call, pinned inputs, H2D + forward + D2H of the logits inside the timed region.  The host submits
    # into `--e2e-inflight` workspace slots (default 3): one more than the device-side measurement, so that the blocking wait for a
    # slot's previous step (its pinned logits must be final before the slot is re-used) does not starve the GPU of submissions.
    enfl = args.e2e_inflight if args.e2e_inflight > 0 else (nfl + 1 if nfl > 1 else 1)
    if args.no_graph:
        enfl = 1
    estreams = streams + [torch.cuda.Stream(device=dev) for _ in range(enfl - len(streams))] if enfl > 1 else [torch.cuda.current_stream(dev)]
    hreqs = [[t.pin_memory() for i, t in enumerate(r) if i != 6] for r in reqs]
    houts = [{"vil_prediction": torch.empty(B, 3129, dtype=torch.float32).pin_memory()} for _ in range(enfl)]
    out_bytes = houts[0]["vil_prediction"].numel() * 4

    def estep(i):
        # host-buffer C-ABI call on slot/stream i % enfl: H2D of this step's inputs, forward, D2H of its logits -- all inside
        # the timed region.  A slot is re-used only after its previous step has completed (its pinned logits are final then),
        # so with several slots one batch's copies overlap another batch's kernels.
        q, f, s, seg, im, vm, tk = hreqs[i % args.rotate]
        j = i % enfl
        if enfl == 1:
            return model.forward_host(q, f, s, seg, im, vm, tk, houts[0], select=L.OUT_VIL_PREDICTION)
        estreams[j].synchronize()
        with torch.cuda.stream(estreams[j]):
            model.forward_host(q, f, s, seg, im, vm, tk, houts[j], select=L.OUT_VIL_PREDICTION, slot=j, synchronize=False)

    def esync():
        for st_ in estreams:
            st_.synchronize()
        torch.cuda.synchronize(dev)

    for i in range(max(args.warmup, 3) * enfl):
        estep(i)
    esync()
    t0 = time.perf_counter()
    for i in range(args.steps):
        estep(i)
    esync()                            # every stream drained: the logits of all steps are in host memory
    e2e_s = time.perf_counter() - t0
    e2e_s = all_rank_ms(e2e_s, world, dev)[0]
    e2e_value = B * world * args.steps / e2e_s
    hout = houts[(args.steps - 1) % enfl]
    chk = model(*dreqs[(args.steps - 1) % args.rotate], select=L.OUT_VIL_PREDICTION)[0].cpu()
    assert torch.allclose(chk, hout["vil_prediction"], atol=1e-5), "host/device C-ABI paths disagree"

    res = dict(value=value, ms=ms, per_rank_ms=per_rank, e2e_value=e2e_value, e2e_s=e2e_s, in_bytes=in_bytes, out_bytes=out_bytes,
               n_launch=int(n_launch), flops=flops, nfl=nfl, enfl=enfl, clocks=sampler.result(), timed_region_s=ms * 1e-3,
               last_out=named_outputs(out))
    if with_profile:
        # ---- per-kernel times, live: every kernel of the step replayed from its own CUDA graph between two CUDA events
        ops = model.profile_ops(B, Tin, V, select, iters=5)
        if args.ops_table:
            agg = {}
            for o in ops:
                k = (o["kind"],) + tuple(o["dims"])
                a_ = agg.setdefault(k, [0, 0.0, 0.0])
                a_[0] += 1; a_[1] += o["ms"]; a_[2] += o["flops"]
            rows = [dict(kind=k[0], dims=list(k[1:]), launches=v[0], total_us=round(v[1] * 1e3, 1), us=round(v[1] * 1e3 / v[0], 2),
                         tflops=round(v[2] / (v[1] * 1e-3) / 1e12, 1) if v[2] else None) for k, v in agg.items()]
            rows.sort(key=lambda r: -r["total_us"])
            with open(args.ops_table, "w") as f:
                for r in rows:
                    f.write(json.dumps(r) + "\n")
        fam = {}
        for o in ops:
            f = fam.setdefault(o["kind"], {"launches": 0, "ms": 0.0, "flops": 0.0})
            f["launches"] += 1; f["ms"] += o["ms"]; f["flops"] += o["flops"]
        res["fam"] = fam
        res["top"] = max((o for o in ops if o["kind"] == "gemm"), key=lambda o: o["flops"])
        # the same GEMM launches with every resident CTA slot as their grid: what a launch does with the GPU to itself
        # (production starts 2/3 of the slots, which is slower alone and faster in the step -- profiles/r2_grid_size.md)
        full = [o for o in model.profile_ops(B, Tin, V, select, iters=5, grid_pct=100) if o["kind"] == "gemm"]
        res["gemm_full_grid_tflops"] = sum(o["flops"] for o in full) / (sum(o["ms"] for o in full) * 1e-3) / 1e12
    return res


def run_vqa(args):
    import torch
    import torch.distributed as dist
    import vilbert_b200 as vb
    from vilbert_b200 import synthetic as S
    from vilbert_b200 import _lib as L

    rank, local_rank, world = env_rank()
    dev = torch.device("cuda", local_rank)
    B, Tin, V = args.batch, args.n_tokens, args.n_regions
    cfg = vb.BertConfig(task_specific_tokens=True, visualization=True)       # worker.py:509-522
    sd = S.synthetic_state_dict(cfg, seed=42)
    select = L.OUT_TASK_HEADS if args.all_heads else L.OUT_VIL_PREDICTION
    # resident inputs: `rotate` distinct batches (8 x 19 MB > 126 MB L2 together with 466 MB of weights)
    reqs = [S.synthetic_request(B, Tin, V, seed=1234 + rank * 1000 + i) for i in range(args.rotate)]
    head = "bf16" if args.dtype == "both" else args.dtype      # BASELINE.json configs[1] names bf16
    alts = ["fp16"] if args.dtype == "both" else []
    oracle = oracle_model(sd, cfg.to_dict(), 3129) if rank == 0 else None
    rows = [0, B // 3, (2 * B) // 3, B - 1]

    model = make_engine(args, sd, cfg, head, local_rank)
    m = measure_vqa(args, model, reqs, dev, world, rank, local_rank, select, with_profile=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, m["last_out"])
    par = parity_rows(model, oracle, reqs[0], rows) if rank == 0 else None
    weight_mb = model._dims["weight_bytes"] / 1e6
    model.close()
    alt = {}
    for dt in alts:
        model = make_engine(args, sd, cfg, dt, local_rank)
        a = measure_vqa(args, model, reqs, dev, world, rank, local_rank, select, with_profile=False)
        ap = parity_rows(model, oracle, reqs[0], rows) if rank == 0 else (None, None)
        model.close()
        alt[dt] = {"value": a["value"], "ms_per_step": a["ms"] / args.steps, "e2e": a["e2e_value"],
                   "max_abs_err_vs_fp32_oracle": ap[0], "logit_std": ap[1], "clocks": a["clocks"]}

    pk = peaks()
    ms, flops, fam, top = m["ms"], m["flops"], m["fam"], m["top"]
    tflops = flops * args.steps / (ms * 1e-3) / 1e12           # per GPU (ms is the max over ranks)
    g = fam["gemm"]
    gemm_tflops = g["flops"] / (g["ms"] * 1e-3) / 1e12
    serial_ms = sum(f["ms"] for f in fam.values())
    traffic = None
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                traffic = json.load(f).get("gemm_dram_bytes_per_launch")
            break
        except Exception:
            pass
    # the whole step is compared with the peak that matches the length of its timed region: a sub-second burst runs at boost
    # clock (burst cuBLAS peak), a seconds-long run sits under the 1000 W cap (sustained peak)
    step_peak = pk["bf16_burst"] if m["timed_region_s"] < 1.0 else pk["bf16_sustained"]
    in_bytes = m["in_bytes"]
    line = {"metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": head, "data": "synthetic",
            "config": {"workload": f"batch={B} per GPU, VQA head, {V} regions x {Tin} tokens (BASELINE.json configs[1]), "
                                   f"{head} tensor-core operands / fp32 accumulate (tcgen05 kind::f16); "
                                   f"random-init 268M-param ViLBERT (seed 42)",
                       "global_batch": B * world, "per_gpu_batch": B, "n_tokens": Tin, "n_regions": V,
                       "parallelism": f"dp{world} (batch sharding, no collective)",
                       "l2": f"inputs rotate over {args.rotate} resident batches ({args.rotate * in_bytes / 1e6:.0f} MB) "
                             f"+ {weight_mb:.0f} MB of weights > 126 MB L2",
                       "batches_in_flight": m["nfl"],
                       "cuda_graph": not args.no_graph, "pdl": "every kernel" if args.pdl != "off" else "off", "layernorm": "fused" if args.fused_ln else "split",
                       "heads": "task heads" if args.all_heads else "vil_prediction"},
            "e2e": {"value": m["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": m["out_bytes"],
                    "ms_per_step": 1e3 * m["e2e_s"] / args.steps, "batches_in_flight": m["enfl"]},
            "gpu_launches": m["n_launch"] * args.steps,
            "launches_per_step": m["n_launch"],
            "parity": {"max_abs_err_vs_fp32_oracle": par[0] if par else None, "logit_std": par[1] if par else None,
                       "rows": rows, "note": "vil_prediction of 4 rows of the timed batch vs the fp32 CPU oracle"},
            "alt": alt,
            "per_rank_ms_per_step": [x / args.steps for x in m["per_rank_ms"]],
            "roofline": {"bound": "tensor", "achieved": gemm_tflops, "peak": pk["bf16_burst"], "unit": "TFLOP/s",
                         "frac": gemm_tflops / pk["bf16_burst"], "traffic": traffic,
                         "kernel": "gemm_persistent_kernel (tcgen05): all %d GEMM launches of one step, algorithmic 2MNK FLOPs / "
                                   "CUDA-event time per launch" % g["launches"],
                         "avg_launch_us": 1e3 * g["ms"] / g["launches"],
                         "largest_gemm": {"M": top["dims"][0], "N": top["dims"][1], "K": top["dims"][2], "us": 1e3 * top["ms"],
                                          "tflops": top["flops"] / (top["ms"] * 1e-3) / 1e12},
                         "achieved_full_grid": m["gemm_full_grid_tflops"], "frac_full_grid": m["gemm_full_grid_tflops"] / pk["bf16_burst"],
                         "grid_note": "achieved/frac: the launches as the step issues them (persistent grid = 2/3 of the 296 CTA slots); "
                                      "*_full_grid: the same launches with all slots, i.e. each kernel alone on the GPU",
                         "share_of_step": g["ms"] / serial_ms,
                         "families_ms": {k: round(v["ms"], 4) for k, v in fam.items()},
                         "whole_step_tflops": tflops, "whole_step_frac": tflops / step_peak,
                         "whole_step_peak": step_peak, "whole_step_frac_vs_burst": tflops / pk["bf16_burst"],
                         "whole_step_frac_vs_sustained": tflops / pk["bf16_sustained"],
                         "flops_per_step": flops,
                         "peak_source": pk["src"] + ": burst cuBLAS bf16 for the kernels timed alone (peak); the whole step against the "
                                        "burst peak when its timed region is < 1 s, else the sustained one (%.0f)" % pk["bf16_sustained"]},
            "clocks": m["clocks"]}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        nb = 3
        times = time_oracle(oracle, reqs[0], nb, 1)
        v = B * len(times) / sum(times)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": CPU_THREADS, "kind": "port",
                                "sample": f"{nb} forwards of batch {B} after 1 warm-up (torch fp32 oracle, "
                                          f"{torch.get_num_threads()} threads of {os.cpu_count()} vCPUs, all heads + pre-training heads)"}
    if rank == 0:
        print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ configs[2]: multi-task
def run_multitask(args):
    """B = batch x world pairs per step, task tokens VQA (1) / NLVR2 (12, adjacent pairs) / RefCOCO (11) in thirds of the GLOBAL batch,
    sharded on pair-aligned boundaries; every rank computes vil_prediction, vil_binary_prediction and vision_logit of its slice."""
    import torch
    import vilbert_b200 as vb
    from vilbert_b200 import parallel as P
    from vilbert_b200 import synthetic as S
    from vilbert_b200 import _lib as L
    rank, local_rank, world = env_rank()
    dev = torch.device("cuda", local_rank)
    Bg, Tin, V = args.batch * world, args.n_tokens, args.n_regions
    cfg = vb.BertConfig(task_specific_tokens=True, visualization=True)
    sd = S.synthetic_state_dict(cfg, seed=42)
    dtype = "bf16" if args.dtype == "both" else args.dtype
    model = make_engine(args, sd, cfg, dtype, local_rank)
    select = L.OUT_VIL_PREDICTION | L.OUT_VIL_BINARY_PREDICTION | L.OUT_VISION_LOGIT
    third = (Bg // 3) // 2 * 2
    tasks = torch.cat([torch.full((third, 1), 1), torch.full((third, 1), 12), torch.full((Bg - 2 * third, 1), 11)]).long()
    lo, hi = P.shard_range(Bg, rank, world, pair_aligned=True)
    reqs = []
    for i in range(args.rotate):
        r = list(S.synthetic_request(Bg, Tin, V, seed=4321 + i))      # the GLOBAL batch (same on every rank), then this rank's slice
        r[7] = tasks
        reqs.append([t[lo:hi].contiguous() for t in r])
    dreqs = [[t.to(dev) for t in r] for r in reqs]
    nfl = max(1, args.inflight)
    streams = [torch.cuda.Stream(device=dev) for _ in range(nfl)] if nfl > 1 else [torch.cuda.current_stream(dev)]

    def step(i):
        if nfl == 1:
            return model(*dreqs[i % args.rotate], select=select)
        with torch.cuda.stream(streams[i % nfl]):
            return model(*dreqs[i % args.rotate], select=select, slot=i % nfl)

    sampler = ClockSampler(local_rank)
    ms_local, out, _ = timed_loop(step, args.steps, args.warmup, streams, dev, world, sampler)
    ms, per_rank = all_rank_ms(ms_local, world, dev)
    sampler.join(timeout=1.0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, named_outputs(out))
    n_launch, flops = model.plan_info(hi - lo, Tin, V, select)
    # parity on this rank's slice: rows re-run alone must give the same bits (shard independence), rank 0 also checks the oracle
    o_all = model(*dreqs[0], select=select)
    pick = [0, (hi - lo) // 2 // 2 * 2]
    o_two = model(*[torch.cat([t[p:p + 2] for p in pick]) for t in dreqs[0]], select=select)
    torch.cuda.synchronize(dev)
    same = all(torch.equal(o_two[0][2 * k:2 * k + 2], o_all[0][p:p + 2]) for k, p in enumerate(pick)) and \
        all(torch.equal(o_two[3][k:k + 1], o_all[3][p // 2:p // 2 + 1]) for k, p in enumerate(pick)) and \
        all(torch.equal(o_two[6][2 * k:2 * k + 2], o_all[6][p:p + 2]) for k, p in enumerate(pick))
    err = None
    if rank == 0:
        oracle = oracle_model(sd, cfg.to_dict(), 3129)
        sub = [torch.cat([t[p:p + 2] for p in pick]) for t in reqs[0]]
        with torch.no_grad():
            torch.set_num_threads(CPU_THREADS)
            ref = oracle(*sub, compute_pretraining_heads=False)
        err = {"vil_prediction": float((o_two[0].cpu() - ref[0]).abs().max()),
               "vil_binary_prediction": float((o_two[3].cpu() - ref[3]).abs().max()),
               "vision_logit": float((o_two[6].cpu() - ref[6]).abs()[ref[6].abs() < 1000].max())}
    ok = torch.tensor([1.0 if same else 0.0], device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    value = Bg * args.steps / (ms * 1e-3)
    if rank == 0:
        line = {"metric": "image-text pairs/sec (multi-task batch: VQA + NLVR2 + RefCOCO heads, 36 regions x 30 tok)", "value": value,
                "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
                "config": {"workload": f"BASELINE.json configs[2]: global batch {Bg} ({args.batch} per GPU), task tokens VQA / NLVR2 / "
                                       f"RefCOCO in thirds, NLVR2 samples as adjacent pairs, pair-aligned contiguous shards, no collective",
                           "global_batch": Bg, "per_gpu_batch": args.batch, "parallelism": f"dp{world}", "batches_in_flight": nfl,
                           "l2": f"inputs rotate over {args.rotate} resident batches"},
                "per_rank_ms_per_step": [x / args.steps for x in per_rank],
                "gpu_launches": int(n_launch) * args.steps, "launches_per_step": int(n_launch),
                "whole_step_tflops_per_gpu": flops * args.steps / (ms * 1e-3) / 1e12,
                "parity": {"shard_rows_bit_identical_on_every_rank": bool(ok.item() == 1.0), "max_abs_err_vs_fp32_oracle": err},
                "clocks": sampler.result()}
        print(json.dumps(line), flush=True)
    model.close()


# ------------------------------------------------------------------------------------------------ configs[3]: retrieval
def run_retrieval(args):
    """score[c, i] = vil_logit of (caption c, image i), task token 7 (worker.py:278-284, 359): captions shard over ranks, every rank
    scores its block against ALL images, one NCCL all-gather (raw ncclAllGather on the compute stream) gives every rank the matrix."""
    import torch
    import torch.distributed as dist
    import vilbert_b200 as vb
    from vilbert_b200 import parallel as P
    from vilbert_b200 import synthetic as S
    from vilbert_b200 import _lib as L
    rank, local_rank, world = env_rank()
    dev = torch.device("cuda", local_rank)
    n_cap, n_img, Tin, V = args.captions, args.images, args.n_tokens, args.n_regions
    cfg = vb.BertConfig(task_specific_tokens=True, visualization=True)
    sd = S.synthetic_state_dict(cfg, seed=42)
    dtype = "bf16" if args.dtype == "both" else args.dtype
    model = make_engine(args, sd, cfg, dtype, local_rank)
    cap = S.synthetic_request(n_cap, Tin, V, seed=7100, full_masks=False)
    img = S.synthetic_request(n_img, Tin, V, seed=7200)
    caps = tuple(cap[i].to(dev) for i in (0, 3, 4))
    imgs = tuple(img[i].to(dev) for i in (1, 2, 5))
    comm = None
    if world > 1:
        from vilbert_b200.nccl_comm import NcclComm
        comm = NcclComm()
    pb = max(args.batch, 64)

    def build(tm=None):
        if args.no_reuse:
            score = P.make_pair_scorer(model, caps, imgs)
            return P.retrieval_scores(score, n_cap, n_img, image_chunk=pb)     # torch.distributed all-gather (baseline path)
        return P.retrieval_scores_cached(model, caps, imgs, pair_batch=pb, comm=comm, timings=tm)

    for _ in range(max(1, min(args.warmup, 1))):
        full = build()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    tms = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0.record()
    for _ in range(args.steps):
        tm = {}
        full = build(tm)
        tms.append(tm)
    e1.record()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    sampler.stop_flag = True
    ms, per_rank = all_rank_ms(e0.elapsed_time(e1), world, dev)
    sampler.join(timeout=1.0)
    assert full.shape == (n_cap, n_img) and torch.isfinite(full).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"scores": full})
    # ---- checks on EVERY rank: (a) the gathered matrix is the same on all ranks, (b) sampled entries, recomputed here with the
    # plain full forward of that pair (no sharding, no reuse), match the matrix bit for bit; rank 0: (c) two entries vs the oracle
    csum = full.double().sum().reshape(1)
    same_everywhere = True
    if world > 1:
        lo_, hi_ = csum.clone(), csum.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        same_everywhere = bool((lo_ == hi_).item())
    g = torch.Generator().manual_seed(99 + rank)
    cs, is_ = torch.randint(0, n_cap, (16,), generator=g), torch.randint(0, n_img, (16,), generator=g)
    task = torch.full((16, 1), 7, dtype=torch.long, device=dev)
    plain = model(caps[0][cs], imgs[0][is_], imgs[1][is_], caps[1][cs], caps[2][cs], imgs[2][is_], None, task, select=L.OUT_VIL_LOGIT)[2].view(-1)
    bit_ok = bool(torch.equal(plain, full[cs.to(dev), is_.to(dev)]))
    okt = torch.tensor([1.0 if bit_ok else 0.0], device=dev)
    if world > 1:
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    err = None
    if rank == 0:
        oracle = oracle_model(sd, cfg.to_dict(), 3129)
        errs = []
        for c, i in ((0, 0), (n_cap - 1, n_img // 2)):
            with torch.no_grad():
                torch.set_num_threads(CPU_THREADS)
                o = oracle(cap[0][c:c + 1], img[1][i:i + 1], img[2][i:i + 1], cap[3][c:c + 1], cap[4][c:c + 1], img[5][i:i + 1], None,
                           torch.full((1, 1), 7), compute_pretraining_heads=False)
            errs.append(abs(float(o[2].view(-1)[0]) - float(full[c, i])))
        err = max(errs)
    pairs = n_cap * n_img
    value = pairs * args.steps / (ms * 1e-3)
    if rank == 0:
        last = tms[-1] if tms and tms[-1] else {}
        line = {"metric": "image-text pairs/sec (caption-image retrieval score matrix, vil_logit, 36 regions x 30 tok)", "value": value,
                "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": 1, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
                "config": {"workload": f"BASELINE.json configs[3]: {n_cap} captions x {n_img} images = {pairs} pair scores, task token 7; "
                                       f"captions sharded contiguously over ranks, "
                                       + ("full forward per pair" if args.no_reuse else
                                          "caption / image prefixes encoded once, connection layers per pair (bit-identical)")
                                       + f", {pb} pairs per forward, ONE all-gather of the fp32 score blocks",
                           "parallelism": f"dp{world} over captions", "collective": "ncclAllGather on the compute stream" if comm else
                           ("none (1 GPU)" if world == 1 else "torch.distributed all_gather_into_tensor")},
                "matrix_seconds": ms * 1e-3 / args.steps,
                "phases_ms_rank0": {k: round(float(v), 3) for k, v in last.items()},
                "all_gather_ms": round(float(last.get("gather_ms", 0.0)), 3) if last else None,
                "all_gather_bytes_per_rank": 4 * (n_cap // world) * n_img if world > 1 else 0,
                "per_rank_ms_per_step": [x / args.steps for x in per_rank],
                "parity": {"matrix_identical_on_all_ranks": same_everywhere,
                           "sampled_entries_equal_plain_forward_bitwise_on_all_ranks": bool(okt.item() == 1.0),
                           "max_abs_err_vs_fp32_oracle_2_entries": err},
                "clocks": sampler.result()}
        print(json.dumps(line), flush=True)
    if comm is not None:
        comm.close()
    model.close()


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank, local_rank, world = env_rank()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the vilbert_b200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        {"vqa": run_vqa, "multitask": run_multitask, "retrieval": run_retrieval}[args.workload](args)
    finally:
        if world > 1:
            dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
