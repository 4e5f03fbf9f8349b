#!/usr/bin/env python
"""bench.py — train tokens/s of a Llama-2-7B NF4+double-quant LoRA finetuning step (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our arm (fused sm_100a Linear4bit), 1 process / GPU
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle dequant + CPU matmul)
  python bench.py --impl unfused ...                       # bnb-equivalent GPU restatement (dequant kernel + cuBLAS)
  python bench.py ... --dump-outputs DIR                   # also save the last timed step's outputs as DIR/*.npy

A "step" = one optimizer step on ONE synthetic OASST-shaped sample per GPU: forward (32 checkpointed decoder
layers, 7 Linear4bit+LoRA each), backward (checkpoint recompute + dX), DDP allreduce of LoRA grads (N>1),
grad-norm clip 0.3, AdamW on the adapters.  Nothing is skipped inside the timed region.
Prints ONE JSON line on rank 0 (contract in the task statement; keys documented in DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "train_tokens_per_sec_llama2_7b_nf4_dq_lora_seq2048"  # for --model/--seq other than the default the name is rebuilt in main()
UNIT = "tokens/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "unfused", "bf16"])
    ap.add_argument("--model", default="llama2-7b")
    ap.add_argument("--seq", type=int, default=2048)
    ap.add_argument("--lora-r", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-baseline-budget-s", type=float, default=0.0, help="deprecated, ignored (the CPU sample always runs all 7 linears)")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the bnb-equivalent GPU restatement timed beside our arm (N=1 only)")
    ap.add_argument("--no-fused-lora", action="store_true", help="keep the LoRA update as separate GEMM + add kernels (peft's form)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying one CUDA graph per step")
    ap.add_argument("--lora-dropout", type=float, default=0.0, help="recipe value 0.1 (scripts/finetune_llama2_guanaco_7b.sh:42); 0 = timing default (SURVEY 8d)")
    ap.add_argument("--grad-accum", type=int, default=1, help="micro-batches per optimizer step (recipe: 16); the gradient allreduce runs on the boundary micro-step only")
    ap.add_argument("--norm-out-fp32", action="store_true", help="reference dtype flow: fp32 norm outputs -> Linear4bit sees fp32 in / returns fp32 (qlora.py:396-405)")
    ap.add_argument("--no-group", action="store_true", help="one launch per Linear4bit instead of grouped q/k/v and gate/up launches")
    ap.add_argument("--optim", default="paged", choices=["torch", "paged"],
                    help="paged (default) = the repo's PagedAdamW32bit (qlora.py:198 optim='paged_adamw_32bit'): capturable, one launch over the "
                         "flat adapter buffer; torch = torch.optim.AdamW(fused, capturable)")
    ap.add_argument("--buckets", type=int, default=1,
                    help="gradient allreduce buckets; > 1 = reverse-layer buckets overlapped with backward on a side stream (DDP's scheme). "
                         "Measured slower than one allreduce after backward at 2 GPUs (96.7 vs 95.3 ms): the NCCL kernels take SMs from "
                         "the persistent NF4 kernel, whose static schedule then needs a second round — see DESIGN.md 5")
    ap.add_argument("--cpu-reps", type=int, default=3, help="repetitions of the CPU sample (median reported)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32): the loss, and a "
                         "fixed seeded sample of the adapter weights after the update and of their clipped gradients")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        # that arm times one decoder layer's Linear4bit path on the host with random packed weights: it runs no training step
        ap.error("--dump-outputs needs a GPU arm (--impl ours, unfused or bf16): --impl reference runs no training step")
    return args


# ---------------------------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md "clocks line")
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu_index), "-lms", "200"], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    smax.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(smax), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU implementation of the path
#   (BASELINE.json configs[0]: "CPU reference via bitsandbytes dequantize_4bit + torch.matmul")
# = oracle C dequantize (split over host threads) + torch CPU matmul, fwd + recompute + dX
# ---------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Physical cores this process may use (SMT siblings only add noise to a GEMM-bound sample)."""
    try:
        import psutil

        phys = psutil.cpu_count(logical=False) or 0
    except Exception:
        phys = 0
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    n = phys if 0 < phys <= avail else avail
    return max(1, n)


class CpuReference:
    """The Linear4bit hot path of ONE decoder layer (all 7 linears x {forward, checkpoint recompute, dX}) on the host:
    the bounded sample of the workload both the `cpu_baseline` object and `--impl reference` time.  Always the same
    work (no time budget, no FLOP scaling), fixed thread count, state built once."""

    def __init__(self, shape, seq: int, threads: int):
        import ctypes as ct
        from concurrent.futures import ThreadPoolExecutor

        import numpy as np
        import torch

        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_c as oc
        from oracle import nf4_oracle as o

        so = os.path.join(ROOT, "oracle", "_build", "libnf4_oracle.so")
        if not os.path.exists(so):
            subprocess.run(["make", "-C", os.path.join(ROOT, "oracle")], check=True, capture_output=True)
        self.lib, self.oc, self.np, self.torch = ct.CDLL(so), oc, np, torch
        torch.set_num_threads(threads)
        self.threads, self.shape, self.seq = threads, shape, seq
        self.code = o.create_dynamic_map()
        self.pool = ThreadPoolExecutor(max_workers=threads)
        h, i = shape.hidden, shape.inter
        self.linears = [(h, h)] * 4 + [(i, h)] * 2 + [(h, i)]  # (N, K)
        rng = np.random.default_rng(0)
        self.states, self.acts = {}, {}
        for n, k in set(self.linears):  # synthetic packed state (random codes are as good as any for timing)
            nelem = n * k
            self.states[(n, k)] = dict(packed=rng.integers(0, 256, nelem // 2, dtype=np.uint8),
                                       q=rng.integers(0, 256, nelem // 64, dtype=np.uint8),
                                       a2=(np.abs(rng.standard_normal((nelem // 64 + 255) // 256)) * 0.01 + 0.01).astype(np.float32),
                                       wbuf=np.empty(nelem, dtype=np.float32))
            self.acts[(n, k)] = (torch.randn(seq, k).to(torch.bfloat16).float(), torch.randn(seq, n).to(torch.bfloat16).float())

    def _dequant(self, n, k):
        st = self.states[(n, k)]
        nblocks = n * k // 64
        chunk = (nblocks + self.threads - 1) // self.threads
        futs = [self.pool.submit(self.oc.dequantize_nested_to_f32, self.lib, st["packed"], st["q"], self.code, st["a2"], 0.02, n * k, 64,
                                 256, lo, min(nblocks, lo + chunk), st["wbuf"]) for lo in range(0, nblocks, chunk)]
        for f in futs:
            f.result()
        return self.torch.from_numpy(st["wbuf"]).view(n, k)

    def layer_seconds(self) -> float:
        torch = self.torch
        t0 = time.perf_counter()
        for n, k in self.linears:
            x, dy = self.acts[(n, k)]
            for _ in range(2):  # forward + checkpoint recompute: dequantize_4bit + F.linear each time
                w = self._dequant(n, k)
                y = (x @ w.t()).to(torch.bfloat16)
            w = self._dequant(n, k)  # backward dX: another full dequant + matmul
            dx = (dy @ w).to(torch.bfloat16)
            del y, dx
        return time.perf_counter() - t0

    def describe(self, reps: int) -> str:
        return (f"Linear4bit hot path of 1 of {self.shape.layers} decoder layers at seq {self.seq}: all 7 linears x (fwd + checkpoint "
                f"recompute + dX) = oracle C dequantize on {self.threads} threads + torch CPU fp32 matmul of bf16-rounded operands; "
                f"median of {reps} runs after 1 warm-up; attention/LoRA/optimizer/lm_head excluded (favours the CPU arm); "
                f"tokens/s = seq / (layers x t_layer)")

    def close(self):
        self.pool.shutdown()


def workload_config(args, world: int) -> dict:
    """`config` of the JSON line — identical for our arm and the reference arm (the workload, not the implementation)."""
    return {"workload": f"{args.model} NF4+double-quant, LoRA r={args.lora_r} alpha=16 dropout={args.lora_dropout} on all 7 linears, "
                        f"seq {args.seq}, bs 1/GPU x grad-accum {args.grad_accum}, grad-checkpointing, AdamW on adapters, clip 0.3",
            "global_batch": world * args.grad_accum, "seq_len": args.seq, "parallelism": f"dp{world}" if world > 1 else "single",
            "l2": "inputs larger than L2 (3.5 GB packed weights streamed every step)"}


def run_reference_arm(args):
    """--impl reference: rank 0 alone times the reference's CPU path on the host cores.  Each of the K steps is ONE bounded
    sample (the Linear4bit hot path of one decoder layer, all 7 linears); `ms_per_step` is the measured time of a sample
    step, `value` the tokens/s of the full model extrapolated from it (x layers; stated in cpu_baseline.sample)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from harness.llama_qlora import SHAPES

    shape = SHAPES[args.model]
    threads = host_threads()
    ref = CpuReference(shape, args.seq, threads)
    for _ in range(max(1, min(args.warmup, 2))):
        ref.layer_seconds()
    t_all0 = time.perf_counter()
    times = [ref.layer_seconds() for _ in range(max(args.steps, 1))]
    wall = time.perf_counter() - t_all0
    ref.close()
    t_layer = statistics.median(times)
    value = args.seq / (t_layer * shape.layers)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": ref.describe(len(times)),
                         "t_layer_s": {"median": t_layer, "min": min(times), "max": max(times)}, "host_count": 1},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
        "note": "one host runs this arm whatever --gpus says (rank 0 only): the value does not scale with N; ms_per_step is the "
                "measured sample step (1 decoder layer's Linear4bit path), the full-model step would be x layers",
        "ms_per_full_step_extrapolated": 1e3 * t_layer * shape.layers,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
# GPU arms
# ---------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 22   # sampled elements per dumped array: 16 MB as float32, so the files stay well under 64 MB in all


def dump_outputs(out_dir: str, loss, params, grads) -> None:
    """What a training step hands back to its caller: the loss, the adapter weights after the optimizer update and the
    gradients the update applied, clipped to norm 0.3 (`grads`: laid out like `params`).  With --grad-accum the loss is the
    last micro-batch's, divided by the micro-batch count as it was backpropagated.  Llama-2-7B has 160 M adapter values, so
    larger outputs are sampled at positions drawn from a fixed seed: the same positions in every run, for element-wise
    comparison."""
    import numpy as np
    import torch

    weights = torch.cat([p.detach().reshape(-1) for p in params])
    n = weights.numel()
    if n <= DUMP_SAMPLE:
        idx = torch.arange(n, device=weights.device)
    else:
        idx = torch.randint(0, n, (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).unique().to(weights.device)
    os.makedirs(out_dir, exist_ok=True)
    out = {"loss": loss.detach().reshape(1), "lora_weights": weights[idx], "lora_grads": grads.detach().reshape(-1)[idx]}
    for name, t in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    import qlora_b200 as q
    import harness.llama_qlora as H
    from harness.llama_qlora import SHAPES, LlamaQLoRA, count_linear4bit_flops, synthetic_batch
    from qlora_b200 import _lib
    from qlora_b200 import autograd as qauto
    from qlora_b200 import functional as QF

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py GPU arms need a GPU (use --impl reference for the CPU path)"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    _lib.load()  # fail loudly if the CUDA extension is missing
    qauto.USE_FUSED = args.impl == "ours"
    from qlora_b200 import lora as qlora_mod

    qlora_mod.ACCUMULATE_ADAPTER_GRADS_IN_PLACE = True   # persistent flat .grad buffers + explicit sync (harness/dp.py)
    H.GROUP_LINEARS = args.impl == "ours" and not args.no_group and not args.no_fused_lora

    shape = SHAPES[args.model]
    accum = max(1, args.grad_accum)
    torch.backends.cuda.matmul.allow_tf32 = True  # qlora.py:70
    # lora_A, embed_tokens and lm_head are initialised from the global RNG: seed it so that every run, and every rank, starts
    # from the same weights
    torch.manual_seed(1234)
    model = LlamaQLoRA(shape, device, lora_r=args.lora_r, lora_alpha=16, lora_dropout=args.lora_dropout, seed=1234,
                       double_quant=True, grad_checkpointing=True, quantized=args.impl != "bf16", norm_out_fp32=args.norm_out_fp32)
    model.train()
    if args.no_fused_lora or args.impl != "ours":
        for mod in model.modules():
            if hasattr(mod, "fused"):
                mod.fused = False
    params = model.trainable_parameters()
    n_lora = sum(p.numel() for p in params)
    if args.optim == "paged":   # qlora.py:198 optim='paged_adamw_32bit' -> bitsandbytes.optim.PagedAdamW32bit (here: the repo's, capturable)
        opt = q.optim.PagedAdamW32bit(params, lr=2e-4, betas=(0.9, 0.999), weight_decay=0.0, capturable=True)
    else:
        opt = torch.optim.AdamW(params, lr=2e-4, betas=(0.9, 0.999), weight_decay=0.0, fused=True, capturable=True)

    # Data parallelism (qlora.py:300-304: one full replica per rank; only the LoRA A/B gradients are reduced).
    # Every LoRA grad is a view into ONE flat bf16 buffer cut into reverse-layer buckets; each bucket's NCCL allreduce starts
    # on a side stream as soon as its layers have finished backward (DDP's overlap), all inside the step's CUDA graph.
    from harness.dp import FlatGradSync

    gsync = FlatGradSync(params, world, layer_of=model.trainable_parameter_layers(), n_buckets=args.buckets, overlap=True,
                         flat_params=args.optim == "paged")
    sync_enabled = [True]
    if world > 1:
        model.layer_backward_done = lambda i: gsync.layer_done(i) if sync_enabled[0] else None

    n_samples = 8
    host_batches = [synthetic_batch(shape, args.seq, seed=1000 * rank + j, pin=True) for j in range(n_samples)]
    dev_batches = [(a.to(device), b.to(device)) for a, b in host_batches]
    static_ids = dev_batches[0][0].clone()
    static_labels = dev_batches[0][1].clone()
    static_loss = torch.zeros((), device=device, dtype=torch.float32)
    clip_coef = torch.ones((), device=device, dtype=torch.float32)

    def micro_body(first: bool, last: bool):
        """One micro-batch: forward + checkpointed backward accumulating into the flat gradient buffer; on the LAST
        micro-batch of the optimizer step also the gradient allreduce, clip 0.3 and AdamW (qlora.py:200 gradient
        accumulation: DDP's no_sync on the others)."""
        if first:
            gsync.zero()
        sync_enabled[0] = last
        model.dropout_seed.add_(1)   # a new dropout mask per micro-batch (no-op for p = 0)
        loss = model(static_ids, static_labels)
        if accum > 1:
            loss = loss / accum
        loss.backward()
        static_loss.copy_(loss.detach())
        if last:
            gsync.finish()
            if args.optim == "paged":
                # --max_grad_norm 0.3: norm over the flat gradient buffer (one kernel), the clip coefficient stays on the
                # device and is applied inside the optimizer kernel (gnorm_scale, as upstream's kernel does)
                torch.clamp(0.3 / (torch.linalg.vector_norm(gsync.flat, dtype=torch.float32) + 1e-6), max=1.0, out=clip_coef)
                opt.step_flat(gsync.flat_param, gsync.flat, grad_scale=clip_coef)   # ONE launch over all 160 M adapter weights
            else:
                torch.nn.utils.clip_grad_norm_(params, 0.3, foreach=True)  # --max_grad_norm 0.3 (scripts/finetune_llama2_guanaco_7b.sh)
                opt.step()

    # warm-up eagerly on a side stream (first-use costs: cuBLAS handles, attention autotune, NCCL rings,
    # cudaFuncSetAttribute of our kernels), then capture the micro-steps into CUDA graphs.
    kinds = [(True, True)] if accum == 1 else [(True, False), (False, False), (False, True)]   # (first, last) variants
    graphs = {}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            for kd in kinds:
                micro_body(*kd)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    use_graph = not args.no_graph
    launches_per_kind = {}
    if use_graph:
        try:
            for kd in kinds:
                QF.LAUNCH_COUNTER[0] = 0
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, capture_error_mode="thread_local"):
                    micro_body(*kd)
                graphs[kd] = g
                launches_per_kind[kd] = QF.LAUNCH_COUNTER[0]   # OUR kernels recorded in this graph = launched per replay
        except Exception as e:  # fall back to eager launches, and say so
            print(f"[bench] CUDA-graph capture failed ({type(e).__name__}: {e}); running eagerly", file=sys.stderr)
            graphs = {}
            use_graph = False
            torch.cuda.synchronize()

    def kind_of(mi: int):
        return (mi == 0, mi == accum - 1)

    def step(batches, j):
        """One optimizer step = `accum` micro-batches (each copies its own inputs into the static buffers)."""
        for mi in range(accum):
            ids, labels = batches[(j * accum + mi) % n_samples]
            static_ids.copy_(ids, non_blocking=True)
            static_labels.copy_(labels, non_blocking=True)
            kd = kind_of(mi)
            if kd in graphs:
                graphs[kd].replay()
            else:
                micro_body(*kd)
        return static_loss

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def timed(loop_fn, n):
        """barrier+sync, CUDA events around n steps, barrier+sync; returns max-over-ranks seconds."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loop_fn(n)
        e1.record()
        barrier()
        secs = torch.tensor([e0.elapsed_time(e1) / 1e3], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(secs, op=dist.ReduceOp.MAX)
        return float(secs.item())

    def loop_resident(n):
        for j in range(n):
            step(dev_batches, j)

    last_loss = [None]

    def loop_e2e(n):
        for j in range(n):
            last_loss[0] = step(host_batches, j).item()     # pinned-host H2D of every micro-batch's inputs ... D2H read of the loss

    loop_resident(max(args.warmup, 3))
    torch.cuda.synchronize()

    if os.environ.get("QB200_NCU_STEP"):  # launch-list capture: `ncu --profile-from-start off ... bench.py`
        torch.cuda.cudart().cudaProfilerStart()
        loop_resident(1)
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        teardown(graphs, world)
        return

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    QF.LAUNCH_COUNTER[0] = 0
    t_res = timed(loop_resident, args.steps)
    if graphs:
        launches = args.steps * sum(launches_per_kind[kind_of(mi)] for mi in range(accum))
    else:
        launches = QF.LAUNCH_COUNTER[0]
    t_e2e = timed(loop_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:   # before the roofline and baseline steps below change the adapters again
        # --optim torch clips the gradient buffer in place; the paged optimizer applies the clip coefficient in its kernel
        dump_outputs(args.dump_outputs, static_loss, params, gsync.flat * clip_coef if args.optim == "paged" else gsync.flat)

    # roofline of the dominant kernel: CUDA events around every fused launch (same stream), a few more micro-steps
    # (launched eagerly: events cannot be recorded inside a replayed graph)
    roof = None
    if args.impl == "ours":
        QF.EVENT_LOG = []
        for j in range(min(args.steps, 3)):
            static_ids.copy_(dev_batches[j % n_samples][0])
            static_labels.copy_(dev_batches[j % n_samples][1])
            micro_body(True, True)
        torch.cuda.synchronize()
        tot_ms, tot_flops, n_l, by_kind = 0.0, 0.0, 0, {}
        for kind, m, n, k, ev0, ev1 in QF.EVENT_LOG:
            ms = ev0.elapsed_time(ev1)
            tot_ms += ms
            tot_flops += 2.0 * m * n * k          # grouped launches log M x problems
            n_l += 1
            d = by_kind.setdefault(f"{kind}:{n}x{k}", [0, 0.0, 0.0])
            d[0] += 1
            d[1] += ms
            d[2] += 2.0 * m * n * k
        log_copy = list(QF.EVENT_LOG)
        QF.EVENT_LOG = None
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = peaks.get("bf16_tflops_sustained")
        peak_src = "measured sustained (MEASURED_PEAKS.json)" if peak else "fallback (B200_PROFILING.md, sustained)"
        peak = peak or 1400.0
        achieved = tot_flops / (tot_ms * 1e-3) / 1e12 if tot_ms > 0 else 0.0
        # DRAM traffic per launch: launch-mix average of the ncu-measured bytes per launch kind — profiles/r2_traffic_by_kind.json
        traffic, traffic_src = None, None
        try:
            tb = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic_by_kind.json")))
            tot_b, ok = 0.0, bool(log_copy)
            for kind, m, n, k, _e0, _e1 in log_copy:
                key = f"{kind}:{n}x{k}:M{m}"
                if key not in tb["bytes"]:
                    ok = False
                    break
                tot_b += tb["bytes"][key]
            if ok:
                traffic = tot_b / len(log_copy)
                traffic_src = "launch-mix mean of dram__bytes_read+write per launch, ncu --set full (profiles/r2_traffic_by_kind.json)"
        except Exception:
            pass
        roof = {"bound": "tensor", "kernel": "nf4_gemm_pair_kernel (fused NF4 dequant + tcgen05 GEMM + LoRA step; grouped q/k/v and gate/up, fwd + dX)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_unit": "bytes/launch", "traffic_source": traffic_src, "peak_source": peak_src,
                "launches_timed": n_l, "avg_launch_us": 1e3 * tot_ms / max(n_l, 1),
                "by_kind": {kk: {"launches": v[0], "avg_us": 1e3 * v[1] / v[0], "tflops": v[2] / (v[1] * 1e-3) / 1e12} for kk, v in by_kind.items()}}

    # The reference's GPU path restated on the same model in the same process (N=1 only): bitsandbytes is not installable
    # here, so this is OUR bit-exact dequantize kernel writing bf16 W to HBM + cuBLAS, with peft's separate LoRA GEMMs —
    # the kernel sequence of SURVEY.md 3.2 (K3+K4 -> K5).  Re-captured as its own CUDA graph.
    gpu_baseline = None
    if args.impl == "ours" and world == 1 and not args.no_gpu_baseline and accum == 1:
        try:
            qauto.USE_FUSED = False
            H.GROUP_LINEARS = False
            for mod in model.modules():
                if hasattr(mod, "fused"):
                    mod.fused = False
            for _ in range(2):
                micro_body(True, True)
            torch.cuda.synchronize()
            g2 = None
            if graphs:
                g2 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g2, capture_error_mode="thread_local"):
                    micro_body(True, True)
            nb = max(3, min(args.steps, 5))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for j in range(nb):
                static_ids.copy_(dev_batches[j % n_samples][0])
                static_labels.copy_(dev_batches[j % n_samples][1])
                if g2 is not None:
                    g2.replay()
                else:
                    micro_body(True, True)
            e1.record()
            torch.cuda.synchronize()
            tb = e0.elapsed_time(e1) / 1e3
            gpu_baseline = {"value": args.seq * nb / tb, "unit": UNIT, "ms_per_step": 1e3 * tb / nb, "steps": nb,
                            "kind": "restatement: bit-exact dequantize kernel (bf16 W written to HBM) + cuBLAS GEMM per Linear4bit call, "
                                    "LoRA as separate GEMMs (peft form); real bitsandbytes is not installable in this image"}
            del g2
        except Exception as e:
            gpu_baseline = {"unavailable": f"{type(e).__name__}: {e}"}
        finally:
            qauto.USE_FUSED = True

    tokens = args.seq * world * args.steps * accum
    value = tokens / t_res
    e2e = tokens / t_e2e
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": 1e3 * t_res / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "config": workload_config(args, world),
        "details": {"impl": args.impl,
                    "lora": ("fused into the NF4 GEMM (extra bf16 k-step)" + ("" if args.no_group else "; q/k/v and gate/up as grouped launches"))
                    if (args.impl == "ours" and not args.no_fused_lora) else "separate GEMMs (peft form)",
                    "launch": "one CUDA graph replay per micro-step" if graphs else "eager launches",
                    "grad_sync": ((f"{len(gsync.buckets)} reverse-layer buckets, NCCL allreduce(AVG) overlapped with backward on a side stream"
                                   if len(gsync.buckets) > 1 else "one flat-buffer NCCL allreduce(AVG) of the LoRA grads after backward")
                                  if world > 1 else "none (1 GPU)"),
                    "optimizer": "qlora_b200.optim.PagedAdamW32bit (capturable, one launch over the flat adapter buffer; clip coefficient applied in the kernel)" if args.optim == "paged"
                    else "torch.optim.AdamW(fused, capturable)",
                    "norm_out": "fp32 (reference dtype flow)" if args.norm_out_fp32 else "bf16", "lora_params": n_lora},
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": 2 * args.seq * 8 * world * accum, "d2h_bytes_per_step": 4 * world,
                "ms_per_step": 1e3 * t_e2e / args.steps, "last_loss": last_loss[0]},
        "gpu_launches": launches, "clocks": clocks,
        "linear4bit_tflops_in_step": 3 * count_linear4bit_flops(shape, args.seq) * world * args.steps * accum / t_res / 1e12,
    }
    if args.impl != "ours":
        line["impl"] = args.impl
    if roof is not None:
        line["roofline"] = roof
    if gpu_baseline is not None:
        line["bnb_equivalent_gpu_baseline"] = gpu_baseline
    if world > 1:
        dist.barrier(device_ids=[local_rank])
    torch.cuda.synchronize()
    if rank == 0:
        if args.impl == "ours" and world == 1 and not args.no_cpu_baseline:
            threads = host_threads()
            ref = CpuReference(shape, args.seq, threads)
            ref.layer_seconds()   # warm-up
            ts = [ref.layer_seconds() for _ in range(max(1, args.cpu_reps))]
            ref.close()
            t_layer = statistics.median(ts)
            line["cpu_baseline"] = {"value": args.seq / (t_layer * shape.layers), "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": ref.describe(len(ts)), "t_layer_s": {"median": t_layer, "min": min(ts), "max": max(ts)}}
        emit(line)
    teardown(graphs, world)


def teardown(graphs, world):
    """Orderly exit (round 1 hard-exited with os._exit, which skipped every atexit hook, the driver's loaded-library record
    included): drop the captured graphs, drain the device, destroy the process group, then return normally.  A watchdog
    turns a teardown that hangs (NCCL communicator destruction with graphs in flight has done so) into a normal-looking
    exit: it runs the atexit hooks itself and only then leaves."""
    import atexit
    import gc

    import torch
    import torch.distributed as dist

    sys.stdout.flush()
    sys.stderr.flush()

    def _bail():
        try:
            atexit._run_exitfuncs()
        finally:
            os._exit(0)

    timer = threading.Timer(45.0, _bail)
    timer.daemon = True
    timer.start()
    graphs.clear()
    gc.collect()
    torch.cuda.synchronize()
    if world > 1 and dist.is_initialized():
        try:
            dist.barrier()
            torch.cuda.synchronize()
            dist.destroy_process_group()
        except Exception as e:
            print(f"[bench] process-group teardown: {type(e).__name__}: {e}", file=sys.stderr)
    timer.cancel()


def count_fused_launches_per_step(shape):
    """Our kernels per training step: every Linear4bit runs forward, checkpoint-recompute forward and dX."""
    return 3 * 7 * shape.layers


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, written to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    global METRIC, _REAL_STDOUT
    # Third-party banners (NCCL version line, torchrun notes, ...) must not share stdout with the JSON line:
    # keep the original stdout for emit() and point fd 1 at stderr for everything else.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse_args()
    METRIC = f"train_tokens_per_sec_{args.model.replace('-', '_')}_nf4_dq_lora_seq{args.seq}"
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
