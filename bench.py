#!/usr/bin/env python
"""Headline benchmark: DeepFM on Criteo-shaped synthetic data, samples/s of the whole job.

Reference benchmark being reproduced: test/benchmark/criteo_deepctr.py (DeepFM via DeepCTR,
26 sparse + 13 dense features, Adagrad, batch 4096 per GPU, embedding dim 9 or 64) whose
published numbers are in BASELINE.md (8x T4). Contract: see the task description --
``python bench.py --gpus N --steps K --warmup W`` prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PUBLISHED_KIPS = {  # BASELINE.md section 1/2, "OpenEmbedding + Horovod" (Cache Local), 8x T4
    ("deepfm", 64): {1: 188, 2: 329, 4: 519, 8: 587},
    ("deepfm", 9): {1: 293, 2: 458, 4: 726, 8: 935},
    ("wdl", 64): {1: 216, 2: 368, 4: 558, 8: 645},
    ("wdl", 9): {1: 308, 2: 476, 4: 683, 8: 935},
    ("xdeepfm", 9): {1: 42, 2: 95, 4: 191, 8: 342},
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=1000)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--impl", default="ours", choices=["ours", "reference", "baseline"],
                   help="ours: this framework; reference: the unmodified reference (unavailable offline); baseline: the same "
                        "model/config/data in plain PyTorch -- NCCL all_to_all + all_reduce, cuBLAS (benchmarks/nccl_baseline.py)")
    p.add_argument("--baseline-dtype", default="bf16", choices=["bf16", "fp32"], help="dense compute dtype of --impl baseline")
    p.add_argument("--model", default="deepfm", choices=["lr", "wdl", "deepfm", "xdeepfm", "dcn"])
    p.add_argument("--dim", type=int, default=64)
    p.add_argument("--batch", type=int, default=4096, help="per-GPU batch (weak scaling)")
    p.add_argument("--vocab", default="criteo1tb_20m", choices=["criteo1tb_20m", "kaggle", "tiny"])
    p.add_argument("--optimizer", default="adagrad", help="sparse AND dense optimizer (adagrad | adam | ftrl, like the reference "
                   "benchmark's --optimizer); other sparse optimizers keep Adagrad on the dense side")
    p.add_argument("--cache", type=int, default=4096, help="replicate tables smaller than this (reference --cache)")
    p.add_argument("--no-graph", action="store_true")
    p.add_argument("--engine", default="auto", choices=["auto", "fused", "eager"],
                   help="fused: every kernel of the step is ours (tcgen05 GEMMs ...); eager: torch dense ops")
    p.add_argument("--allreduce", default="auto")
    p.add_argument("--skew", type=float, default=1.0, help="0 = uniform ids, 1 = log-uniform (Zipf-like)")
    p.add_argument("--pool", type=int, default=16, help="distinct pre-generated batches cycled through")
    p.add_argument("--no-prefetch", action="store_true",
                   help="do not announce the next batch's ids one step ahead (default: the public prefetch API, the reference's "
                        "pulling(): the next batch's pull + plan run beside this step's dense all-reduce / optimizer)")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write what the last device-timed step computed as DIR/<name>.npy (float32, rank 0): its loss, "
                        "the dense parameters after its update and the embedding rows of its batch read back after it")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs covers --impl ours")
    return a


DUMP_PARAMS = 4 << 20           # floats of dense parameters, at most (16 MB)
DUMP_ROWS_BYTES = 32 << 20      # bytes of embedding rows, at most: a dump stays under 64 MB


def _sample_rows(torch, t, n, seed):
    """``t`` if it has at most ``n`` rows, else ``n`` of its rows (in order, with repeats) picked by a fixed seed"""
    if t.shape[0] <= n:
        return t
    g = torch.Generator(device="cpu").manual_seed(seed)
    idx = torch.randint(t.shape[0], (n,), generator=g).sort().values
    return t[idx.to(t.device)]


def dump_outputs(torch, model, loss, ids):
    """What a training step computed, as float32 host arrays: ``loss`` (what ``step`` returns), the dense parameters
    after its update (flat, in the model's order; replicated small tables included) and the server-side embedding
    rows of its batch ``ids`` read back by a stateless pull ([batch, io_stride], the model's activation layout;
    columns no server table feeds are 0). Larger outputs are cut to a seeded sample of rows."""
    dense = model.theta if hasattr(model, "theta") else torch.cat([p.detach().reshape(-1) for p in model.dense_parameters()])
    out = {"loss": loss.detach().reshape(1), "dense_params": _sample_rows(torch, dense, DUMP_PARAMS, 1)}
    if model.sparse is not None:
        rows = torch.zeros((ids.shape[0], model.sparse.io_stride), dtype=torch.float32, device=ids.device)
        rows = model.sparse.group.pull(ids, out=rows)
        out["embedding_rows"] = _sample_rows(torch, rows, max(1, DUMP_ROWS_BYTES // (4 * rows.shape[1])), 2)
    return {k: v.float().cpu().numpy() for k, v in out.items()}


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = str(gpu_index), [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 9 and f[0] == self.idx:
                self.rows.append(f)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for j, n in enumerate(names):
                if r[5 + j].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def make_batches(torch, vocab, n_dense, batch, pool, skew, seed, device):
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    out = []
    v = torch.tensor(vocab, dtype=torch.float64)
    for _ in range(pool):
        u = torch.rand((batch, len(vocab)), generator=g, dtype=torch.float64)
        if skew > 0:
            ids = torch.floor(torch.exp(u * torch.log(v))) - 1            # log-uniform: P(id<=x) ~ log x
            ids = ids.clamp_(min=0)
        else:
            ids = torch.floor(u * v)
        ids = ids.to(torch.int64)
        vv = torch.tensor(vocab, dtype=torch.int64)
        ids = (ids * 2654435761 + 12345) % vv                              # scatter hot ids over shards
        dense = torch.rand((batch, n_dense), generator=g, dtype=torch.float32)
        labels = (torch.rand((batch,), generator=g) < 0.25).to(torch.float32)
        out.append((ids.pin_memory(), dense.pin_memory(), labels.pin_memory()))
    return out


def run_baseline(a, torch, dist, world, rank, local_rank):
    """--impl baseline: plain PyTorch (NCCL + cuBLAS) arm, same metric / config / data / timing rules."""
    from benchmarks.nccl_baseline import HostPipeline, NcclBaselineCTR
    from openembedding_b200.models.ctr import CRITEO_1TB_VOCAB_20M, CRITEO_KAGGLE_VOCAB   # constants only
    vocab = {"criteo1tb_20m": CRITEO_1TB_VOCAB_20M, "kaggle": CRITEO_KAGGLE_VOCAB,
             "tiny": [min(v, 10007) for v in CRITEO_KAGGLE_VOCAB]}[a.vocab]
    dev = torch.device("cuda", local_rank)
    assert a.model in ("deepfm", "wdl") and a.optimizer == "adagrad", "the baseline arm covers DeepFM / WDL with Adagrad"
    cdt = torch.bfloat16 if a.baseline_dtype == "bf16" else torch.float32
    model = NcclBaselineCTR(vocab, num_dense=13, embedding_dim=a.dim, model=a.model, batch=a.batch,
                            cache_threshold=a.cache, compute_dtype=cdt, rank=rank, world=world, device=dev)
    host = make_batches(torch, vocab, 13, a.batch, a.pool, a.skew, 1000 + rank, dev)
    devb = [(i.to(dev), d.to(dev), l.to(dev)) for i, d, l in host]

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for s in range(a.warmup):
        model.step(*devb[s % a.pool])
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for s in range(a.steps):
        loss = model.step(*devb[(a.warmup + s) % a.pool])
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    loss_val = float(loss)
    pipe = HostPipeline(model, a.batch, len(vocab), 13)
    for s in range(max(3 * getattr(pipe, "NBUF", 1), a.warmup // 2)):      # every (buffer i -> buffer i+1) graph variant exists before timing
        pipe.submit(*host[s % a.pool])
    pipe.last_loss()
    sync_all()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for s in range(a.steps):
        pipe.submit(*host[(a.warmup + s) % a.pool])
    e2e_loss = pipe.last_loss()
    f1.record()
    sync_all()
    t = torch.tensor([ms, f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        gb = a.batch * world
        pub = PUBLISHED_KIPS.get((a.model, a.dim), {}).get(world)
        value = gb * a.steps / (ms / 1e3)
        rows = sum(vocab)
        print(json.dumps({
            "impl": "baseline",
            "metric": "samples/sec (whole job, device-timed, max over ranks) %s Criteo dim %d" % (a.model, a.dim),
            "value": value, "unit": "samples/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (value / (pub * 1e3)) if pub else None, "dtype": a.baseline_dtype,
            "data": "synthetic (Criteo-shaped: 26 sparse log-uniform ids + 13 dense, random-init weights)",
            "config": {"model": "%s (DeepCTR architecture), emb dim %d, adagrad sparse / Adagrad dense" % (a.model, a.dim),
                       "global_batch": gb, "seq_len": 1,
                       "parallelism": "dp%d + row-sharded embeddings (id %% %d): NCCL all_to_all ids/rows/grads + NCCL all_reduce" % (world, world),
                       "vocab_rows_total": rows, "cache_threshold": a.cache, "cuda_graph": False,
                       "engine": "plain PyTorch: torch.unique + index ops, torch.nn / cuBLAS (%s), torch.distributed NCCL" % a.baseline_dtype,
                       "l2_policy": "inputs larger than L2: %d distinct random batches" % a.pool},
            "clocks": clocks,
            "e2e": {"value": gb * a.steps / (e2e_ms / 1e3), "unit": "samples/s", "h2d_bytes_per_step": pipe.h2d_bytes,
                    "d2h_bytes_per_step": pipe.d2h_bytes, "ms_per_step": e2e_ms / a.steps},
            "gpu_launches": 0, "nccl_calls_per_step": model.nccl_calls / max(1, a.warmup + 2 * a.steps + max(3, a.warmup // 2)),
            "final_loss": loss_val, "e2e_final_loss": e2e_loss}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    a = parse()
    if a.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:      # launched under torchrun for N > 1: one line, from rank 0
            return 0
        print(json.dumps({"impl": "reference", "unavailable":
                          "offline install failed: setup.py needs the CMake-generated openembedding_setup + prebuilt "
                          "libcexb_pack.so (~20 third-party C++ libs fetched by URL) and TensorFlow 2.x + Horovod, "
                          "none of which are in the image/wheelhouse (see DESIGN.md)"}))
        return 0
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        print(json.dumps({"error": "bench.py needs a CUDA device"}))
        return 1
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert world == a.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"

    if a.impl == "baseline":
        return run_baseline(a, torch, dist, world, rank, local_rank)
    import openembedding_b200 as oe
    from openembedding_b200 import _native
    from openembedding_b200.context import get_context
    from openembedding_b200.models.ctr import CRITEO_1TB_VOCAB_20M, CRITEO_KAGGLE_VOCAB, CTRModel
    from openembedding_b200.models.trainer import Trainer
    oe.flags.device = "cuda"
    ctx = get_context()
    vocab = {"criteo1tb_20m": CRITEO_1TB_VOCAB_20M, "kaggle": CRITEO_KAGGLE_VOCAB,
             "tiny": [min(v, 10007) for v in CRITEO_KAGGLE_VOCAB]}[a.vocab]
    torch.manual_seed(1234)
    engine = a.engine
    if engine == "auto":
        engine = "fused" if (a.model in ("deepfm", "wdl") and a.batch % 128 == 0) else "eager"
    dense_opt = {"category": a.optimizer if a.optimizer in ("adagrad", "adam", "ftrl") else "adagrad"}
    if engine == "fused":
        from openembedding_b200.models.fused_dense import FusedCTR, FusedTrainer
        model = FusedCTR(vocab, num_dense=13, embedding_dim=a.dim, model=a.model, batch=a.batch,
                         sparse_optimizer={"category": a.optimizer}, cache_threshold=a.cache, dense_optimizer=dense_opt)
        trainer = FusedTrainer(model, use_graph=not a.no_graph)
        trainer.want_prefetch = not a.no_prefetch
    else:
        model = CTRModel(vocab, num_dense=13, embedding_dim=a.dim, model=a.model, batch=a.batch,
                         sparse_optimizer={"category": a.optimizer}, cache_threshold=a.cache)
        trainer = Trainer(model, use_graph=not a.no_graph, allreduce=a.allreduce, dense_optimizer=dense_opt)
    dev = ctx.device
    host = make_batches(torch, vocab, 13, a.batch, a.pool, a.skew, 1000 + rank, dev)
    devb = [(i.to(dev), d.to(dev), l.to(dev)) for i, d, l in host]

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    prefetch = engine == "fused" and not a.no_prefetch

    def run_step(k):
        if prefetch:      # public prefetch API: the ids of the NEXT batch are announced one step ahead (reference: pulling())
            # stable=True: the pool's device tensors stay alive at fixed addresses (graphs are captured on them)
            return trainer.step(*devb[k % a.pool], next_ids=devb[(k + 1) % a.pool][0], stable=True)
        return trainer.step(*devb[k % a.pool])

    # ---------------- device-timed headline number
    if prefetch and not a.no_graph:
        for s in range(a.pool + 2):     # untimed set-up, before the W warm-up steps: one graph per resident batch of the pool
            run_step(s)
    for s in range(a.warmup):
        run_step(s)
    sync_all()
    ctx.backend.engine.check()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for s in range(a.steps):
        loss = run_step(a.warmup + s)
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    loss_val = float(loss)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    ctx.backend.engine.check()
    dumped = dump_outputs(torch, model, loss, devb[(a.warmup + a.steps - 1) % a.pool][0]) if a.dump_outputs else None

    # ---------------- end-to-end through the public pipeline API: pinned H2D in, loss D2H out, every step
    pipe = trainer.make_pipeline(a.batch, len(vocab), 13)
    for s in range(max(3 * getattr(pipe, "NBUF", 1), a.warmup // 2)):      # every (buffer i -> buffer i+1) graph variant exists before timing
        pipe.submit(*host[s % a.pool])
    pipe.last_loss()
    sync_all()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    f0.record()
    for s in range(a.steps):
        pipe.submit(*host[(a.warmup + s) % a.pool])
    e2e_loss = pipe.last_loss()
    f1.record()
    sync_all()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max(f0.elapsed_time(f1), 0.0)
    t = torch.tensor([e2e_ms, wall_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t[0])
    clocks = sampler.stop() if rank == 0 else None     # sampled over both timed regions (device-timed + end-to-end)
    ctx.backend.engine.check()

    if rank == 0:
        gb = a.batch * world
        value = gb * a.steps / (ms / 1e3)
        e2e_value = gb * a.steps / (e2e_ms / 1e3)
        pub = PUBLISHED_KIPS.get((a.model, a.dim), {}).get(world)
        if engine == "fused":
            own_kernels_per_step = model.kernels_per_step()
        else:
            own_kernels_per_step = 2 + (5 if (world > 1 and trainer._ar is not None) else 0)
        rows = sum(vocab)
        line = {
            "metric": "samples/sec (whole job, device-timed, max over ranks) %s Criteo dim %d" % (a.model, a.dim),
            "value": value, "unit": "samples/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (value / (pub * 1e3)) if pub else None,
            "dtype": "bf16", "data": "synthetic (Criteo-shaped: 26 sparse log-uniform ids + 13 dense, random-init weights)",
            "config": {"model": "%s (DeepCTR architecture), emb dim %d, %s sparse / %s dense" % (a.model, a.dim, a.optimizer, dense_opt["category"]),
                       "global_batch": gb, "seq_len": 1, "parallelism": "dp%d + row-sharded embeddings (id %% %d) over NVLink" % (world, world),
                       "vocab_rows_total": rows, "tables_fp32_gb": round(rows * (a.dim + 1) * 4 * 2 / 2 ** 30, 1),
                       "cache_threshold": a.cache, "cuda_graph": not a.no_graph, "engine": engine, "prefetch": prefetch,
                       "sparse_kernels": ("v2 (planned batch, pre-reduced push)" if getattr(getattr(model, "group", None), "v2", False)
                                          else "v1 (stateless pull, dispatch/combine push)") if engine == "fused" else "v1 (eager layers)",
                       "dense_allreduce": ("none (1 GPU)" if world == 1 else
                                           "inside the sparse push kernel" if getattr(model, "_rider", False) else
                                           "stand-alone P2P kernel"),
                       "l2_policy": "inputs larger than L2: %d distinct random batches over a %.0f GB table working set" % (
                           a.pool, rows * (a.dim + 1) * 8 / 2 ** 30)},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": pipe.h2d_bytes,
                    "d2h_bytes_per_step": pipe.d2h_bytes, "ms_per_step": e2e_ms / a.steps, "wall_ms_per_step": wall_ms / a.steps},
            "gpu_launches": own_kernels_per_step * a.steps,
            "native_libs": {"cuda": _native.cuda_loaded()},
            "final_loss": loss_val, "e2e_final_loss": e2e_loss,
            "push_update_phases_us": ctx.backend.engine.status()[1].get("last_push_update_us"),
            "pull_probe_us": [round((x - ctx.backend.engine.status()[1]["probe"][0]) / 1e3, 2) if x else None
                              for x in ctx.backend.engine.status()[1]["probe"][:8]],
            "sparse_counters": {k: v for k, v in ctx.backend.engine.status()[1].items()
                                if k in ("pull_indices", "pull_unique", "push_indices", "update_unique",
                                         "nvlink_rows_pulled", "nvlink_rows_pushed", "plans")},
        }
        print(json.dumps(line))
        if dumped is not None:
            import numpy as np
            os.makedirs(a.dump_outputs, exist_ok=True)
            for name, arr in dumped.items():
                np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
