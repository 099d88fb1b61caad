#!/usr/bin/env python
"""Headline benchmark: UNITER-base encoder fwd+bwd samples/s (BASELINE.json configs[1] = C2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dtype bf16|fp16]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic batch per GPU: H2D (e2e leg only),
UniterModel forward (embeddings + 12 BertLayers on packed tokens) + MLM head + loss, backward,
and for N > 1 the gradient allreduce (NCCL, mean) — weak scaling, 64 samples per GPU.
Prints ONE JSON line on rank 0 (contract in the task statement; extra keys: roofline,
cpu_baseline, clocks, e2e, gpu_launches, breakdown).

`--dump-outputs DIR` writes what the last timed step computed (see dump_outputs) so that two
builds can be compared output for output: the inputs, weights and dropout seeds are fixed, so the
same arguments give the same inputs on every run.

`--impl reference` times the CPU restatement of the reference path (oracle/, kind "port" — the
reference is Python and cannot travel to the GPU box) on the host cores, bounded sample.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "uniter_base_encoder_fwd_bwd_samples_per_sec"
BASE = dict(vocab=28996, H=768, NL=12, heads=12, I=3072, max_pos=512, img_dim=2048)
LARGE = dict(vocab=28996, H=1024, NL=24, heads=16, I=4096, max_pos=512, img_dim=2048)
C2 = dict(B=64, tl=(12, 28), nbb=(26, 46), seed=1234, mlm_prob=0.15)
# BASELINE.json configs (SURVEY.md §8d).  The default (and the driver's) run is C2, the config the
# metric is quoted on; the others are reachable with --config for the profiles / docs.
CONFIGS = {
    "c3": dict(label="C3"),
    "c5": dict(label="C5"),
    "c2": dict(label="C2", arch=BASE, arch_name="UNITER-base", metric=METRIC, tasks=("mlm",),
               B=64, tl=(12, 28), nbb=(26, 46), seed=1234, mlm_prob=0.15, mrm_prob=0.15),
    "c4": dict(label="C4", arch=LARGE, arch_name="UNITER-large",
               metric="uniter_large_pretrain_fwd_bwd_samples_per_sec",
               tasks=("mlm", "mrfr", "mrc-kl", "itm"),
               B=64, tl=(12, 28), nbb=(26, 46), seed=1234, mlm_prob=0.15, mrm_prob=0.15),
}
IMG_LABEL_DIM = 1601


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--cpu-sample", type=int, default=64,
                    help="samples in the CPU arm's batch (64 = the full C2 batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--overlap-chunks", type=int, default=4,
                    help="N>1: layer groups whose gradient all-reduce overlaps the backward pass")
    ap.add_argument("--sm-reserve", type=int, default=0,
                    help="N>1: SMs left to the overlapped all-reduce (and its CTA cap)")
    ap.add_argument("--no-graph", action="store_true",
                    help="enqueue every step from Python (eager) instead of replaying CUDA graphs")
    ap.add_argument("--allreduce", default="peer", choices=["after", "split", "in-graph", "peer"],
                    help="N>1: 'peer' (default) = the gradient slices are exchanged over NVLink peer memory by the "
                         "library itself (csrc/peer.cu: copy-engine transfers + flag / local-reduction kernels) as nodes "
                         "of the step's ONE graph, overlapped with the backward; falls back to 'after' if the start-up "
                         "self-test fails or a flag wait expires; "
                         "'after' = NCCL all-reduce of the arena after each replay; 'split' = the step is "
                         "captured as one graph per layer group and each group's slice is all-reduced (eagerly, on a "
                         "side stream) while the next group's graph runs; 'in-graph' = NCCL captured inside the graph "
                         "(split / in-graph: experimental, not re-measured since captures became local events)")
    ap.add_argument("--peer-ctas", type=int, default=-1,
                    help="--allreduce peer: form of the exchange that overlaps the backward: -1 = copy engines move the "
                         "bytes, SMs only reduce locally; 0 = push + reduce kernels of short-lived CTAs; N > 0 = one "
                         "persistent kernel of N CTAs")
    ap.add_argument("--peer-tail-ctas", type=int, default=-1,
                    help="--allreduce peer: the same for the exchange kernels issued after the backward")
    ap.add_argument("--token-bucket", type=int, default=128,
                    help="graph mode: token counts are padded to a multiple of this with a dummy sequence")
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS),
                    help="c2 (default, the metric's config): UNITER-base MLM; c4: UNITER-large 24-layer "
                         "pre-training step, tasks cycled mlm -> mrfr -> mrc-kl -> itm; c3: UNITER-base VQA fine-tuning, 5 accumulated "
                         "micro-batches of <= 5120 padded tokens; c5: UNITER-base ITM "
                         "hard-negative iteration (400-pair no-grad scoring + 32-pair train step, both directions)")
    ap.add_argument("--layers", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss and the gradients of the last timed step as "
                         "DIR/<name>.npy (float32 / float64, a fixed sample of each large gradient); the GPU "
                         "arm only (--impl ours)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU arm computed (--impl ours)")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.config == "c5" and int(os.environ.get("WORLD_SIZE", "1")) > 1 and args.steps % 8:
        ap.error("c5 on N > 1 GPUs: --steps must be a multiple of 8 (one all-reduce per 8 iterations)")
    return args


DUMP_SAMPLE = 1 << 16      # entries kept of each larger gradient: ~21 MB in all for c2 / c3 / c5, ~40 MB for c4


def dump_outputs(out_dir, loss, model):
    """What a caller of the timed step receives from its last step: the loss (loss.npy; c5: the
    text->images and image->texts losses) and every parameter gradient, zeros for a parameter the
    step left without one.  A gradient of at most DUMP_SAMPLE entries is written whole as
    grad.<parameter>.npy; of a larger one, the entries of the flattened gradient at DUMP_SAMPLE indices
    torch.randint draws from a CPU generator seeded with the first 8 hex digits of the parameter
    name's SHA-1.  grad_norms.npy holds the float64 L2 norm of each full gradient, in
    named_parameters() order."""
    import hashlib
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    if isinstance(loss, (list, tuple)):
        loss = torch.stack([l.reshape(()) for l in loss])
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    norms = []
    for name, p in model.named_parameters():
        g = (p.grad if p.grad is not None else torch.zeros_like(p)).detach().reshape(-1)
        norms.append(g.double().norm().item())
        if g.numel() > DUMP_SAMPLE:
            seed = int(hashlib.sha1(name.encode()).hexdigest()[:8], 16)
            idx = torch.randint(0, g.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(seed))
            g = g[idx.to(g.device)]
        np.save(os.path.join(out_dir, "grad.%s.npy" % name), g.float().cpu().numpy())
    np.save(os.path.join(out_dir, "grad_norms.npy"), np.array(norms, dtype=np.float64))


def algorithmic_flops(lens, NL, H):
    """SURVEY.md §8d: F_fwd+bwd = 3 * NL * (24 H^2 T + 4 H sum S^2), valid tokens only."""
    T = sum(lens)
    s2 = sum(s * s for s in lens)
    return 3.0 * NL * (24.0 * H * H * T + 4.0 * H * s2)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            j = json.load(fh)
        return dict(tflops=j["bf16_tflops"], tflops_sustained=j.get("bf16_tflops_sustained"),
                    hbm_gbs=j["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0,
                source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# =============================================================================== CPU (reference) arm
def _probe_threads(one_step):
    """"all the host threads it can use": torch's CPU GEMMs on these small matrices get SLOWER when
    oversubscribed (128 threads: 0.2 samples/s vs 8 threads: ~20), so probe upwards and keep the
    fastest thread count — the honest best case for the CPU arm."""
    ncpu = os.cpu_count() or 1
    best_t, best_n = None, 1
    for n in [c for c in (4, 8, 16, 32, 64, 128, 256) if c <= ncpu] or [ncpu]:
        torch.set_num_threads(n)
        t = one_step()
        if best_t is None or t < best_t:
            best_t, best_n = t, n
        elif t > 1.5 * best_t:
            break
    torch.set_num_threads(best_n)
    return best_n


def peer_selftest(dev):
    """Start-up check of the NVLink peer-memory exchange (collective): cudaIpc mapping works on this
    box and three all-reduces of a small buffer give the NCCL result.  (ok, reason) — identical on
    every rank, so that all ranks take the same path."""
    import torch.distributed as dist
    from uniter_b200 import distributed as ubd
    ok, why = 1.0, ""
    try:
        n = 8 << 20                     # 16 MB: its own cudaMalloc segment of the caching allocator
        flat = torch.zeros(n, device=dev, dtype=torch.bfloat16)
        px = ubd.PeerExchange(flat, timeout_ms=3000)
        g = torch.Generator(device=dev).manual_seed(7 + dist.get_rank())
        for rep in range(3):
            flat.copy_(torch.randn(n, device=dev, generator=g).to(torch.bfloat16))
            want = flat.float()
            dist.all_reduce(want, op=dist.ReduceOp.SUM)
            want = (want / dist.get_world_size()).to(torch.bfloat16)
            px.all_reduce(0, n)
            torch.cuda.synchronize()
            if px.error_word() != 0:
                ok, why = 0.0, "flag wait expired"
                break
            if not torch.allclose(flat.float(), want.float(), rtol=8e-3, atol=1e-6):
                ok, why = 0.0, "wrong result"
                break
        px.close()
    except Exception as e:            # mapping refused (no peer access / ipc disabled in this container)
        ok, why = 0.0, "%s: %s" % (type(e).__name__, str(e)[:120])
    t = torch.tensor([ok], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if t.item() != 1.0 and not why:
        why = "failed on another rank"
    return t.item() == 1.0, why


def cpu_reference_run(args, steps, warmup, sample_B):
    """The reference's OWN path on the host cores: `UniterForPretraining.forward(batch, 'mlm')`
    (model/pretrain.py:107-133 over model/model.py:336-367) fwd+bwd of the mean MLM loss, fp32,
    train mode (dropout 0.1), on the padded [B, L] rectangle exactly as the reference computes it.
    Runs the UNMODIFIED reference modules staged in oracle/_ref (kind "reference"); only when they
    are absent, the clean-room oracle port (kind "port")."""
    from oracle import ref_loader
    from uniter_b200.synth import seeded_state, synth_batch
    NL = args.layers or BASE["NL"]
    full = synth_batch(C2["B"], C2["tl"][0], C2["tl"][1], C2["nbb"][0], C2["nbb"][1], C2["seed"],
                       mlm_prob=C2["mlm_prob"])
    if sample_B >= C2["B"]:
        sample_B, batch = C2["B"], full
    else:
        tl, nb = full["txt_lens"][:sample_B], full["num_bbs"][:sample_B]
        batch = synth_batch(sample_B, 0, 0, 0, 0, C2["seed"], txt_lens=tl, num_bbs=nb, mlm_prob=C2["mlm_prob"])
    T = sum(a + b for a, b in zip(batch["txt_lens"], batch["num_bbs"]))
    kind = ref_loader.kind()
    if kind == "reference":
        rm, rpre = ref_loader.load("model.model", "model.pretrain")
        cfg = rm.UniterConfig(BASE["vocab"], hidden_size=BASE["H"], num_hidden_layers=NL,
                              num_attention_heads=BASE["heads"], intermediate_size=BASE["I"],
                              max_position_embeddings=BASE["max_pos"])
        torch.manual_seed(0)
        model = rpre.UniterForPretraining(cfg, BASE["img_dim"], 1601).train()
        ref_batch = {k: v for k, v in batch.items() if torch.is_tensor(v)}

        def one_step():
            model.zero_grad()
            t0 = time.perf_counter()
            loss = model(ref_batch, task="mlm", compute_loss=True).mean()
            loss.backward()
            return time.perf_counter() - t0
    else:
        from oracle import encoder_oracle as orc
        from uniter_b200.synth import uniter_state_shapes
        shapes = {"uniter." + k: v for k, v in uniter_state_shapes(BASE["H"], NL, BASE["I"], BASE["vocab"],
                                                                    BASE["max_pos"], 2, BASE["img_dim"]).items()}
        shapes.update({"cls.predictions.transform.dense.weight": (BASE["H"], BASE["H"]),
                       "cls.predictions.transform.dense.bias": (BASE["H"],),
                       "cls.predictions.transform.LayerNorm.weight": (BASE["H"],),
                       "cls.predictions.transform.LayerNorm.bias": (BASE["H"],),
                       "cls.predictions.bias": (BASE["vocab"],)})
        state = {k: v.requires_grad_(True) for k, v in seeded_state(shapes, seed=0).items()}

        def one_step():
            for v in state.values():
                v.grad = None
            t0 = time.perf_counter()
            loss = orc.mlm_forward(state, NL, BASE["heads"], batch).mean()
            loss.backward()
            return time.perf_counter() - t0

    best_n = _probe_threads(one_step)
    times = [one_step() for _ in range(warmup + steps)]
    t = sum(times[warmup:]) / max(1, steps)
    what = ("all %d C2 samples" % sample_B) if sample_B == C2["B"] else \
        ("first %d of the %d C2 samples" % (sample_B, C2["B"]))
    return dict(value=sample_B / t, ms_per_step=t * 1e3, cores=best_n, host_cores=os.cpu_count() or 1,
                kind=kind, batch=sample_B,
                sample="%s (T=%d valid tokens, padded rectangle), %d timed fwd+bwd steps after %d warm-up, "
                       "fp32, dropout 0.1, %s; %d torch threads (fastest of a 4..%d probe) on %d host cores"
                       % (what, T, steps, warmup,
                          "UNMODIFIED reference UniterForPretraining('mlm') from oracle/_ref" if kind == "reference"
                          else "oracle port (reference sources not staged)",
                          best_n, os.cpu_count() or 1, os.cpu_count() or 1))


# =============================================================================== C3: VQA fine-tuning
def bench_c3(args, real_out, rank, world, local_rank):
    """BASELINE.json configs[2]: UNITER-base VQA fine-tuning with the shapes of
    config/train-vqa-base-4gpu.json (train_vqa.py:183-229): per GPU a micro-batch of <= 5120 PADDED
    tokens with a sample count that is a multiple of 8 (TokenBucketSampler, data/sampler.py:31-57),
    text 5..22 tokens + 10..100 regions, 3129 answers, soft targets; 5 micro-batches are accumulated
    per optimizer step and the gradients all-reduced once (gradient_accumulation_steps = 5).
    One STEP here = those 5 micro-batches (fwd + bwd each, accumulated in the gradient arena) + the
    all-reduce for N > 1.  Each micro-batch is a CUDA-graph replay (first: overwrite, others:
    accumulate); the VQA classifier (model/vqa.py:23-28) is torch over the library pooler."""
    import random
    import torch.distributed as dist
    from torch.nn import functional as F
    from uniter_b200 import _lib
    from uniter_b200 import distributed as ubd
    from uniter_b200.arena import GradArena
    from uniter_b200.batching import TokenBucketSampler
    from uniter_b200.graphed import GraphedStep
    from uniter_b200.heads import UniterForVisualQuestionAnswering
    from uniter_b200.model import UniterConfig
    from uniter_b200.synth import synth_batch

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    _lib.check(lib.ub200_device_check())
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    NA, ACC, MAXTOK = 3129, 5, 5120
    torch.manual_seed(0)
    NLr = args.layers or BASE["NL"]
    cfg = UniterConfig(BASE["vocab"], hidden_size=BASE["H"], num_hidden_layers=NLr,
                       num_attention_heads=BASE["heads"], intermediate_size=BASE["I"],
                       max_position_embeddings=BASE["max_pos"])
    model = UniterForVisualQuestionAnswering(cfg, BASE["img_dim"], NA).to(dev, dtype).train()
    if world > 1:
        ubd.broadcast_parameters(model, root=0)
    GradArena.attach(model)
    reducer = ubd.GradientReducer(model, overlap_chunks=1) if world > 1 else None

    # a pool of examples with the config's length ranges, batched by the reference's own sampler logic
    g = torch.Generator().manual_seed(1000 + rank)
    n_pool = 2048
    tls = torch.randint(5, 23, (n_pool,), generator=g).tolist()
    nbs = torch.randint(10, 101, (n_pool,), generator=g).tolist()
    lens_pool = [a + b for a, b in zip(tls, nbs)]
    batches = list(iter(TokenBucketSampler(lens_pool, bucket_size=8192, batch_size=MAXTOK, droplast=True,
                                           rng=random.Random(7 + rank))))
    host = []
    for ids in batches[:ACC]:
        b = synth_batch(len(ids), 0, 0, 0, 0, seed=300 + len(host), txt_lens=[tls[i] for i in ids],
                        num_bbs=[nbs[i] for i in ids])
        b["targets"] = torch.rand(len(ids), NA, generator=g)
        hb = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in b.items()}
        hb["lens"] = [tls[i] + nbs[i] for i in ids]
        host.append(hb)
    samples_per_step = sum(len(h["lens"]) for h in host)
    h2d_bytes = sum(v.numel() * v.element_size() for hb in host for v in hb.values() if torch.is_tensor(v))

    def loss_fn(batch):
        # train_vqa.py:186-188: loss.mean() * num_answers, divided over the accumulation window by the
        # optimizer step (delay_unscale) — here folded into the loss
        l = model(batch, compute_loss=True)
        return l.float().mean() * NA / ACC

    step = GraphedStep(model, loss_fn)
    dev_batches = [{k: v.to(dev, non_blocking=True) for k, v in hb.items() if torch.is_tensor(v)} for hb in host]
    torch.cuda.synchronize()

    def one_step(i, from_host=False):
        for j, hb in enumerate(host):
            src = {k: v for k, v in hb.items() if torch.is_tensor(v)} if from_host else dev_batches[j]
            loss = step(src, hb["lens"], accumulate=j > 0)
        if reducer is not None:
            reducer.reduce()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    for i in range(max(3, args.warmup)):
        one_step(i)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last_loss = [None]

    def timed_step(i):
        last_loss[0] = one_step(i)

    ms_res = timed(timed_step, args.steps) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_loss[0], model)
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()

    def e2e(i):
        l = one_step(i, from_host=True)          # H2D of every micro-batch from pinned memory, in stream
        loss_host.copy_(l.float().reshape(1), non_blocking=True)

    for i in range(2):
        e2e(i)
    ms_e2e = timed(e2e, args.steps) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        flops = sum(algorithmic_flops(h["lens"], NLr, BASE["H"]) for h in host)
        pk = peaks()
        launches = sum(b.launches for b in step.buckets.values()) // 2
        line = {
            "metric": "uniter_base_vqa_finetune_samples_per_sec",
            "value": round(samples_per_step * world / (ms_res * 1e-3), 1), "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms_res, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic",
            "config": {"workload": "C3: UNITER-base VQA fine-tuning (train-vqa-base-4gpu.json shapes): %d "
                                   "micro-batches of <= 5120 padded tokens (%s samples, text 5..22 + 10..100 "
                                   "regions, %d valid tokens) accumulated per step, 3129 answers, dropout 0.1"
                                   % (ACC, "+".join(str(len(h["lens"])) for h in host),
                                      sum(sum(h["lens"]) for h in host)),
                       "global_batch": samples_per_step * world, "parallelism": "dp%d" % world},
            "e2e": {"value": round(samples_per_step * world / (ms_e2e * 1e-3), 1), "unit": "samples/s",
                    "ms_per_step": round(ms_e2e, 4), "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
            "step_mode": "cuda_graph per micro-batch (%d graphs), all-reduce after the window" % step.captures,
            "gpu_launches": int(launches),
            "algorithmic_tflops_per_step": round(flops / 1e12, 4),
            "achieved_tflops": round(flops / (ms_res * 1e-3) / 1e12, 1),
            "roofline": {"bound": "tensor", "kernel": "whole step (encoder GEMMs dominate)",
                         "achieved": round(flops / (ms_res * 1e-3) / 1e12, 1), "peak": pk["tflops"],
                         "unit": "TFLOP/s", "frac": round(flops / (ms_res * 1e-3) / 1e12 / pk["tflops"], 4),
                         "peak_source": pk["source"], "traffic": None},
            "clocks": clocks,
        }
        print(json.dumps(line), file=real_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


# =============================================================================== C5: ITM hard negatives
def bench_c5(args, real_out, rank, world, local_rank):
    """BASELINE.json configs[4]: UNITER-base ITM with in-batch hard negatives
    (train_itm_hard_negatives.py:165-199, model/itm.py:57-147).  One ITERATION = text->images
    (1 text x 400 images: no-grad eval forward of 400 pairs, top-31 hardest, train fwd+bwd of 32
    pairs) followed by the image->texts mirror; `train_batch_size` = 8 iterations accumulate into
    the gradient arena before one all-reduce (config/train-itm-coco-base-16gpu-hn.json).
    Reported: encoder sequences/s ((400 + 32) x 2 per iteration, all ranks) and the reference's
    own counter hn_per_s (hard examples = 32 x 2 per iteration, train_itm_hard_negatives.py:230-237).
    Eager (the hard-negative mining is data dependent: one small device->host read per direction,
    where the reference reads too, model/itm.py:113)."""
    import torch.distributed as dist
    from uniter_b200 import _lib
    from uniter_b200 import distributed as ubd
    from uniter_b200.arena import GradArena
    from uniter_b200.batching import hard_neg_batch_from_image, hard_neg_batch_from_text
    from uniter_b200.heads import UniterForImageTextRetrievalHardNeg
    from uniter_b200.model import UniterConfig, register_lengths

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    _lib.check(lib.ub200_device_check())
    lib.ub200_launch_count.restype = C.c_ulonglong
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    NEG, HARD, TBS, NBB, D = 399, 31, 8, 36, BASE["img_dim"]
    torch.manual_seed(0)
    cfg = UniterConfig(BASE["vocab"], hidden_size=BASE["H"], num_hidden_layers=args.layers or BASE["NL"],
                       num_attention_heads=BASE["heads"], intermediate_size=BASE["I"],
                       max_position_embeddings=BASE["max_pos"])
    model = UniterForImageTextRetrievalHardNeg(cfg, D, margin=0.2, hard_size=HARD).to(dev, dtype).train()
    model.init_output()
    if world > 1:
        ubd.broadcast_parameters(model, root=0)
    GradArena.attach(model)
    reducer = ubd.GradientReducer(model, overlap_chunks=1) if world > 1 else None

    g = torch.Generator().manual_seed(4321 + rank)

    def boxes(n):
        xy = torch.rand(n, 4, generator=g)
        x1 = torch.minimum(xy[:, 0], xy[:, 2]); x2 = torch.maximum(xy[:, 0], xy[:, 2])
        y1 = torch.minimum(xy[:, 1], xy[:, 3]); y2 = torch.maximum(xy[:, 1], xy[:, 3])
        return torch.stack([x1, y1, x2, y2, x2 - x1, y2 - y1, (x2 - x1) * (y2 - y1)], 1)

    def text():
        tl = int(torch.randint(8, 63, (1,), generator=g))
        ids = torch.randint(1000, BASE["vocab"], (tl,), generator=g)
        ids[0], ids[-1] = 101, 102
        return ids

    def make_iteration():
        bt = hard_neg_batch_from_text(text(), [torch.randn(NBB, D, generator=g) for _ in range(NEG + 1)],
                                      [boxes(NBB) for _ in range(NEG + 1)])
        bi = hard_neg_batch_from_image(torch.randn(NBB, D, generator=g), boxes(NBB),
                                       [text() for _ in range(NEG + 1)])
        out = []
        for b in (bt, bi):
            hb = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in b.items()}
            out.append(hb)
        return out

    n_host = 3
    host = [make_iteration() for _ in range(n_host)]
    h2d_bytes = sum(v.numel() * v.element_size() for it in host for hb in it for v in hb.values()
                    if torch.is_tensor(v)) // n_host
    seqs_per_iter = 2 * (NEG + 1 + HARD + 1)

    def to_device(hb):
        d = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in hb.items()}
        register_lengths(d["attn_masks"], [a + b for a, b in zip(hb["txt_lens"], hb["num_bbs"])], prefix=True)
        return d

    copy_stream = torch.cuda.Stream()
    nxt = {}

    def prefetch(i):
        """H2D of iteration i's two batches on a copy stream while iteration i-1 computes
        (data/loader.py:107-138)."""
        copy_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(copy_stream):
            nxt["pair"] = [to_device(hb) for hb in host[i % n_host]]

    def iteration(i, resident=None):
        if resident is not None:
            pair = resident
        else:
            torch.cuda.current_stream().wait_stream(copy_stream)
            pair = nxt["pair"]
            for b in pair:
                for t in b.values():
                    if torch.is_tensor(t):
                        t.record_stream(torch.cuda.current_stream())
            prefetch(i + 1)
        if i % TBS == 0:
            model.zero_grad(set_to_none=True)
        losses = []
        for b, sf in zip(pair, ("t", "i")):
            loss = model(dict(b), sample_from=sf, compute_loss=True).mean() / TBS
            loss.backward()
            losses.append(loss.detach())
        if (i + 1) % TBS == 0 and reducer is not None:
            reducer.reduce()
        return losses

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    steps = args.steps
    resident = [to_device(hb) for hb in host[0]]
    for i in range(max(args.warmup, 3)):
        iteration(i, resident)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.ub200_launch_count()
    last_loss = [None]

    def timed_it(i):
        last_loss[0] = iteration(i, resident)

    ms_res = timed(timed_it, steps) / steps
    launches = (lib.ub200_launch_count() - launches0) // steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_loss[0], model)
    prefetch(0)
    for i in range(n_host):
        iteration(i)
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()

    def e2e_it(i):
        ls = iteration(i)
        if (i + 1) % TBS == 0:
            loss_host.copy_(ls[0].float().reshape(1), non_blocking=True)

    ms_e2e = timed(lambda i: e2e_it(n_host + i), steps) / steps
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        lens_t = [a + b for a, b in zip(host[0][0]["txt_lens"], host[0][0]["num_bbs"])]
        lens_i = [a + b for a, b in zip(host[0][1]["txt_lens"], host[0][1]["num_bbs"])]
        NLr = args.layers or BASE["NL"]
        f_fwd = (algorithmic_flops(lens_t, NLr, BASE["H"]) + algorithmic_flops(lens_i, NLr, BASE["H"])) / 3.0
        f_train = 2 * 3.0 * NLr * (24.0 * BASE["H"] ** 2 * 32 * (sum(lens_t) / 400.0)
                                   + 4.0 * BASE["H"] * 32 * (sum(lens_t) / 400.0) ** 2)
        pk = peaks()
        flops_iter = f_fwd + f_train
        line = {
            "metric": "uniter_base_itm_hardneg_encoder_sequences_per_sec",
            "value": round(seqs_per_iter * world / (ms_res * 1e-3), 1), "unit": "sequences/s",
            "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_res, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic",
            "config": {"workload": "C5: UNITER-base ITM hard negatives; per iteration text->400 images and "
                                   "image->400 texts (36 regions, text 8..62 tokens, S <= 98): no-grad eval "
                                   "forward of 400 pairs, top-31 + positive = 32-pair train fwd+bwd each; "
                                   "8 iterations per all-reduce; rank-0 batch T = %d / %d valid tokens"
                                   % (sum(lens_t), sum(lens_i)),
                       "global_batch": seqs_per_iter * world, "parallelism": "dp%d" % world},
            "hn_per_s": round(2 * (HARD + 1) * world / (ms_res * 1e-3), 1),
            "e2e": {"value": round(seqs_per_iter * world / (ms_e2e * 1e-3), 1), "unit": "sequences/s",
                    "ms_per_step": round(ms_e2e, 4), "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
            "step_mode": "eager (data-dependent hard-negative mining)",
            "gpu_launches": int(launches),
            "algorithmic_tflops_per_step": round(flops_iter / 1e12, 4),
            "achieved_tflops": round(flops_iter / (ms_res * 1e-3) / 1e12, 1),
            "roofline": {"bound": "tensor", "kernel": "whole iteration (encoder GEMMs dominate)",
                         "achieved": round(flops_iter / (ms_res * 1e-3) / 1e12, 1), "peak": pk["tflops"],
                         "unit": "TFLOP/s", "frac": round(flops_iter / (ms_res * 1e-3) / 1e12 / pk["tflops"], 4),
                         "peak_source": pk["source"], "traffic": None},
            "clocks": clocks,
        }
        print(json.dumps(line), file=real_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


# =============================================================================== our arm
def main():
    args = parse()
    # exactly ONE line on stdout: libraries that print there (NCCL's version banner does) are
    # diverted to stderr at the file-descriptor level; the JSON line goes to the saved descriptor
    sys.stdout.flush()
    out_fd = os.dup(1)
    os.dup2(2, 1)
    real_out = os.fdopen(out_fd, "w")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        nst = args.steps
        r = cpu_reference_run(args, nst, 1, args.cpu_sample)
        cb = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "host_cores": r["host_cores"],
              "kind": r["kind"], "sample": r["sample"]}
        line = {"metric": METRIC, "value": r["value"], "unit": "samples/s", "impl": "reference",
                "n_gpus": args.gpus, "steps": nst, "warmup": 1,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "C2: UNITER-base %d-layer encoder fwd+bwd + MLM head (15%% text masked), "
                                       "B=%d, the reference's own CPU path (%s), train mode dropout 0.1"
                                       % (args.layers or BASE["NL"], r["batch"], r["kind"]),
                           "global_batch": r["batch"], "parallelism": "cpu"},
                "cpu_baseline": cb,
                "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}}
        print(json.dumps(line), file=real_out, flush=True)
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    if args.config == "c5":
        return bench_c5(args, real_out, rank, world, local_rank)
    if args.config == "c3":
        return bench_c3(args, real_out, rank, world, local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from uniter_b200 import _lib
    from uniter_b200.arena import GradArena
    from uniter_b200.graphed import GraphedStep
    from uniter_b200.model import UniterConfig, register_lengths
    from uniter_b200.heads import UniterForMLM
    from uniter_b200.synth import pad_mlm_index, synth_batch
    from uniter_b200 import distributed as ubd

    lib = _lib.load()
    _lib.check(lib.ub200_device_check())
    lib.ub200_launch_count.restype = C.c_ulonglong
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    CF = CONFIGS[args.config]
    ARCH = CF["arch"]
    NL = args.layers or ARCH["NL"]
    tasks = CF["tasks"]

    torch.manual_seed(0)
    cfg = UniterConfig(ARCH["vocab"], hidden_size=ARCH["H"], num_hidden_layers=NL,
                       num_attention_heads=ARCH["heads"], intermediate_size=ARCH["I"],
                       max_position_embeddings=ARCH["max_pos"])
    if tasks == ("mlm",):
        model = UniterForMLM(cfg, ARCH["img_dim"])
    else:
        from uniter_b200.heads import UniterForPretraining
        model = UniterForPretraining(cfg, ARCH["img_dim"], IMG_LABEL_DIM)
    model = model.to(device=dev, dtype=dtype).train()
    if world > 1:
        ubd.broadcast_parameters(model, root=0)
    GradArena.attach(model)          # one flat gradient buffer: head | pooler | layers | front-end
    peer_note = None
    if world > 1 and args.allreduce == "peer":
        ok, why = peer_selftest(dev)
        if not ok:
            peer_note = "peer exchange self-test failed (%s): NCCL all-reduce after each replay instead" % why
            args.allreduce = "after"
            if rank == 0:
                print("bench: " + peer_note, file=sys.stderr)
    reducer = (ubd.GradientReducer(model, overlap_chunks=args.overlap_chunks, sm_reserve=args.sm_reserve,
                                   transport="peer" if args.allreduce == "peer" else "nccl",
                                   peer_ctas=args.peer_ctas, peer_tail_ctas=args.peer_tail_ctas)
               if world > 1 else None)

    # ---- synthetic batches (per-rank seed), host side pinned; masked-token / masked-region lists are
    # padded to a multiple of 64 so that every batch of a token bucket replays the same graph.
    # One task per step, cycled (what MetaLoader does, data/loader.py:39-57).
    from uniter_b200.synth import synth_mrm
    n_host = 4 * len(tasks)
    host = []
    for i in range(n_host):
        task = tasks[i % len(tasks)]
        if i < len(tasks):
            # the canonical batch of the config (SURVEY.md §8d: seed 1234 -> T = 3451).  Weak scaling means
            # the SAME work on every GPU: every rank uses the canonical LENGTH profile (so no rank is the
            # straggler of the synchronous step just because it drew longer sequences) with its own token
            # ids / region features / masks.
            b = synth_batch(CF["B"], CF["tl"][0], CF["tl"][1], CF["nbb"][0], CF["nbb"][1],
                            CF["seed"], mlm_prob=CF["mlm_prob"])
            canon = (b["txt_lens"], b["num_bbs"])
            if rank > 0:
                b = synth_batch(CF["B"], 0, 0, 0, 0, CF["seed"] + 1000 * rank,
                                txt_lens=canon[0], num_bbs=canon[1], mlm_prob=CF["mlm_prob"])
        else:
            # further host batches of the rotation: the SAME length profile (so that the e2e leg does
            # the same work per step as the resident leg) with different token ids / features / masks
            b = synth_batch(CF["B"], 0, 0, 0, 0, CF["seed"] + 1000 * rank + 7 * (i // len(tasks)),
                            txt_lens=canon[0], num_bbs=canon[1], mlm_prob=CF["mlm_prob"])
        lens = [a + c for a, c in zip(b["txt_lens"], b["num_bbs"])]
        if task == "mlm":
            b = pad_mlm_index(b, 64)
        else:
            b = {k: v for k, v in b.items() if k not in ("txt_labels", "mlm_index", "mlm_targets")}
            if task in ("mrfr", "mrc-kl"):
                b = synth_mrm(b, CF["mrm_prob"], IMG_LABEL_DIM, seed=i, pad_multiple=64)
                for k in ("img_mask_tgt", "feat_targets" if task != "mrfr" else "label_targets"):
                    b.pop(k)                                    # only what this task's head reads travels
            elif task == "itm":
                b["targets"] = torch.randint(0, 2, (CF["B"],), generator=torch.Generator().manual_seed(i))
        hb = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in b.items()}
        hb["lens"], hb["task"] = lens, task
        host.append(hb)
    lens0 = host[0]["lens"]
    h2d_bytes = sum(sum(v.numel() * v.element_size() for v in hb.values() if torch.is_tensor(v))
                    for hb in host) // n_host

    def loss_fn(batch, task):
        """The scalar the reference's loop back-propagates: `loss.mean()` (pretrain.py:297) — with
        fixed-size (padded) row lists the padding rows contribute 0 and the divisor is the true count."""
        if task == "mlm":
            per_row = model(batch) if tasks == ("mlm",) else model(batch, "mlm")
            return (per_row.sum() * batch["mlm_inv_n"]).squeeze()
        if task == "mrfr":
            l = model(batch, "mrfr").float()                                  # [n_pad, D]
            return ((l * batch["mrm_valid"].unsqueeze(1)).sum() * batch["mrm_inv_n"] / l.size(1)).squeeze()
        if task == "mrc-kl":
            l = model(batch, "mrc-kl").float()                                # [n_pad, labels]
            return ((l * batch["mrm_valid"].unsqueeze(1)).sum() * batch["mrm_inv_n"] / l.size(1)).squeeze()
        if task == "itm":
            return model(batch, "itm")[0].mean()
        raise ValueError(task)

    # N > 1: the gradient exchange is captured INSIDE the graph (peer transport: memcpy + kernel nodes on a
    # side stream, overlapped with the backward); --allreduce after keeps it out of the graph and issues
    # NCCL all-reduces after each replay (the fallback if the peer self-test fails or a flag wait expires)
    ar_mode = "none" if reducer is None else args.allreduce
    graphed = None
    if not args.no_graph:
        graphed = GraphedStep(model, loss_fn, token_bucket=args.token_bucket,
                              reducer=reducer if ar_mode in ("in-graph", "split", "peer") else None,
                              reducer_mode="split" if ar_mode == "split" else "in-graph")

    def replay(bk):
        loss = graphed.replay(bk)
        if ar_mode == "after":
            reducer.reduce()
        return loss

    def to_device(hb, stream):
        with torch.cuda.stream(stream):
            d = {k: v.to(dev, non_blocking=True) for k, v in hb.items() if torch.is_tensor(v)}
        return d

    def eager_step(batch, lens, task):
        register_lengths(batch["attn_masks"], lens, prefix=True)
        model.zero_grad(set_to_none=True)
        loss = loss_fn(batch, task)
        if reducer is not None:
            reducer.backward_and_reduce(loss)
        else:
            loss.backward()
        return loss.detach()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    # (two attempts at most: if a flag wait of the peer exchange expired — a rank-count or topology this
    #  build was never run on — the measurement is repeated with the NCCL all-reduce after each replay)
    for attempt in (0, 1):
        # ---- resident-input measurement ("value"): inputs already in HBM, the step is replayed
        # (one resident batch per task, cycled)
        nt = len(tasks)
        resident = [to_device(host[i], torch.cuda.current_stream()) for i in range(nt)]
        torch.cuda.synchronize()
        if graphed is not None:
            bks = [graphed.stage(resident[i], host[i]["lens"], tag=tasks[i]) for i in range(nt)]   # captures (untimed)
            for i in range(args.warmup):
                replay(bks[i % nt])
            step_resident = lambda i: replay(bks[i % nt])  # noqa: E731
        else:
            for i in range(args.warmup):
                eager_step(resident[i % nt], host[i % nt]["lens"], tasks[i % nt])
            step_resident = lambda i: eager_step(resident[i % nt], host[i % nt]["lens"], tasks[i % nt])  # noqa: E731
        torch.cuda.synchronize()
        launches0 = lib.ub200_launch_count()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        cpu_t = [0.0]
        last_loss = [None]

        def timed_step(i):
            t0 = time.perf_counter()
            last_loss[0] = step_resident(i)
            cpu_t[0] += time.perf_counter() - t0

        ms_total = timed(timed_step, args.steps)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, last_loss[0], model)
        cpu_enqueue_ms = cpu_t[0] / args.steps * 1e3   # host time to enqueue one step (no sync inside)
        if graphed is not None:
            launches = sum(b.launches for b in bks) // nt     # libub200 kernels inside one replay of a graph
        else:
            launches = (lib.ub200_launch_count() - launches0) // args.steps
        ms_step = ms_total / args.steps
        value = CF["B"] * world / (ms_step * 1e-3)

        # ---- e2e: host batches from pinned memory, H2D on a copy stream into rotating device staging
        # buffers while the previous step computes, device-to-device into the graph's static inputs,
        # replay, loss read back asynchronously
        copy_stream = torch.cuda.Stream()
        state = {}

        def prefetch(i):
            hb = host[i % n_host]
            copy_stream.wait_stream(torch.cuda.current_stream())
            state["next"] = (to_device(hb, copy_stream), hb)

        loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
        loss_events = [torch.cuda.Event(), torch.cuda.Event()]
        losses = []
        e2e_cpu, wait = [0.0], [0.0]

        def e2e_step(i):
            t0 = time.perf_counter()
            torch.cuda.current_stream().wait_stream(copy_stream)
            batch, hb = state["next"]
            for t in batch.values():
                t.record_stream(torch.cuda.current_stream())
            if graphed is not None:
                bk = graphed.stage(batch, hb["lens"], tag=hb["task"])
                prefetch(i + 1)
                replay(bk)
                loss = bk.loss
            else:
                prefetch(i + 1)
                loss = eager_step(batch, hb["lens"], hb["task"])
            # D2H read of the step's result: asynchronous copy into pinned memory, consumed while the
            # next step is already enqueued (a blocking .item() here would drain the GPU queue every
            # step, which the reference's own loop does, train_vqa.py:201 — noted, not copied)
            slot = i & 1
            loss_host[slot:slot + 1].copy_(loss.detach().float().reshape(1), non_blocking=True)
            loss_events[slot].record()
            wait[0] = 0.0
            if i > 0:
                tw = time.perf_counter()
                loss_events[slot ^ 1].synchronize()          # the host runs at most one step ahead
                wait[0] = time.perf_counter() - tw
                losses.append(float(loss_host[slot ^ 1]))
            e2e_cpu[0] += time.perf_counter() - t0 - wait[0]

        # warm-up covers every distinct host batch once (each has its own token count: graph buckets are
        # captured / the caching allocator sees its block sizes before the timed region), and the batch
        # rotation continues across the warm-up / timed boundary
        prefetch(0)
        n_warm = max(args.warmup, n_host + 1)
        for i in range(n_warm):
            e2e_step(i)
        e2e_cpu[0] = 0.0
        ms_e2e = timed(lambda i: e2e_step(n_warm + i), args.steps) / args.steps
        e2e_host_ms = e2e_cpu[0] / args.steps * 1e3
        clocks = sampler.stop() if rank == 0 else None     # sampled across both timed regions (under load)
        assert all(l == l for l in losses), "NaN loss in the e2e leg"
        e2e_value = CF["B"] * world / (ms_e2e * 1e-3)
        peer_err = 0
        if reducer is not None and reducer.peer is not None:
            t = torch.tensor([float(reducer.peer.error_word() != 0)], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            peer_err = int(t.item())
        if not peer_err:
            break
        peer_note = ("a flag wait of the NVLink peer exchange expired on this box: re-measured with the NCCL "
                     "all-reduce after each replay")
        if rank == 0:
            print("bench: " + peer_note, file=sys.stderr)
        args.allreduce = ar_mode = "after"
        reducer = ubd.GradientReducer(model, overlap_chunks=args.overlap_chunks, sm_reserve=args.sm_reserve)
        graphed = None if args.no_graph else GraphedStep(model, loss_fn, token_bucket=args.token_bucket, reducer=None)

    def step(i):                                       # eager step for the per-launch event pass
        return eager_step(resident[i % nt], host[i % nt]["lens"], tasks[i % nt])

    # ---- per-kernel-role pass (CUDA events around every launch on the launching stream)
    breakdown, roofline = None, None
    flops_step = sum(algorithmic_flops(host[i]["lens"], NL, ARCH["H"]) for i in range(nt)) / nt
    pk = peaks()
    if not args.no_profile:
        NT = 24
        lib.ub200_profile_enable(1)
        psteps = 3 * nt
        for i in range(psteps):
            step(i)
        ms_arr = (C.c_float * NT)()
        cnt_arr = (C.c_int * NT)()
        _lib.check(lib.ub200_profile_collect(ms_arr, cnt_arr, NT))
        lib.ub200_profile_enable(0)
        names = {0: "gather/cvt", 1: "qkv_gemm", 2: "attn_fwd", 3: "attnout_gemm", 4: "ln1_fwd",
                 5: "ffn1_gemm", 6: "ffn2_gemm", 7: "ln2_fwd", 8: "ln2_bwd", 9: "ffn2_dgrad",
                 10: "wgrad_grouped(4)", 11: "ffn1_dgrad", 12: "ffn1_wgrad", 13: "ln1_bwd",
                 14: "attnout_dgrad", 15: "attnout_wgrad", 16: "attn_bwd", 17: "colsum",
                 18: "qkv_dgrad", 19: "qkv_wgrad", 20: "grad_add"}
        breakdown = {names[i]: {"ms_per_step": round(ms_arr[i] / psteps, 4), "launches": cnt_arr[i] // psteps}
                     for i in range(NT) if cnt_arr[i] > 0}
        gemm_tags = [1, 3, 5, 6, 9, 10, 11, 12, 14, 15, 18, 19]
        gemm_ms = sum(ms_arr[i] for i in gemm_tags) / psteps
        all_ms = sum(ms_arr[i] for i in range(NT)) / psteps       # every library launch, same (serialised) mode
        gemm_launches = sum(cnt_arr[i] for i in gemm_tags) // psteps
        T = sum(sum(host[i]["lens"]) for i in range(nt)) / nt
        gemm_flops = 3.0 * NL * 24.0 * ARCH["H"] ** 2 * T          # dense-projection part of §8d
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tp):                                      # from the committed ncu capture
            with open(tp) as fh:
                tj = json.load(fh)
            traffic = tj["dram_read_bytes_per_launch"] + tj["dram_write_bytes_per_launch"]
            traffic_src = tj["source"]
        achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        roofline = {"bound": "tensor", "kernel": "ub::gemm_kernel (tcgen05, all 12 GEMM roles of a layer)",
                    "achieved": round(achieved, 1), "peak": pk["tflops"], "unit": "TFLOP/s",
                    "frac": round(achieved / pk["tflops"], 4), "peak_source": pk["source"],
                    "launches_per_step": gemm_launches, "avg_launch_us": round(gemm_ms * 1e3 / max(1, gemm_launches), 2),
                    "algorithmic_flops_per_step": gemm_flops, "traffic": traffic, "traffic_unit": "bytes per launch (dram read+write)",
                    "traffic_source": traffic_src,
                    "step_frac_of_peak": round(flops_step / (ms_step * 1e-3) / 1e12 / pk["tflops"], 4),
                    "kernel_time_share_of_step": round(gemm_ms / max(all_ms, 1e-9), 3),
                    "share_basis": "event pass: the 12 GEMM roles / all library launches, both timed launch by "
                                   "launch (serialised); compare with the ncu launch list in profiles/",
                    "event_pass_ms_per_step": round(all_ms, 4)}

    # ---- informational: the same step followed by the fused clip + AdamW update (SURVEY.md §8f-2).
    # NOT part of `value` (BASELINE.json's metric is encoder fwd+bwd); reported beside it.
    train_step = None
    if not args.no_profile and world == 1:
        try:
            from uniter_b200.optim import FusedAdamW
            nd = ("bias", "LayerNorm.bias", "LayerNorm.weight")
            decay = [p for n, p in model.named_parameters() if not any(k in n for k in nd)]
            nodecay = [p for n, p in model.named_parameters() if any(k in n for k in nd)]
            opt = FusedAdamW([{"params": decay, "weight_decay": 0.01}, {"params": nodecay, "weight_decay": 0.0}],
                             lr=1e-6, betas=(0.9, 0.98))

            def opt_step(i):
                step(i)
                opt.step(max_grad_norm=2.0)

            for i in range(3):
                opt_step(i)
            nst = max(5, args.steps // 2)
            ms_opt = timed(opt_step, nst) / nst
            train_step = {"ms_per_step": round(ms_opt, 4),
                          "samples_per_s": round(CF["B"] * world / (ms_opt * 1e-3), 1),
                          "includes": "fwd + bwd + global-norm clip + fused multi-tensor AdamW (fp32 masters)"}
        except Exception as e:      # informational leg: never lose the headline line over it
            train_step = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---- CPU baseline (rank 0, N == 1 only): oracle port on the host cores, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.config == "c2":
        r = cpu_reference_run(args, 2, 1, args.cpu_sample)
        cpu = {"value": round(r["value"], 2), "unit": "samples/s", "cores": r["cores"],
               "host_cores": r["host_cores"], "kind": r["kind"], "sample": r["sample"]}

    if rank == 0:
        line = {
            "metric": CF["metric"], "value": round(value, 1), "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic",
            "config": {"workload": "%s: %s %d-layer encoder fwd+bwd + %s, "
                                   "B=%d per GPU, varlen S~54 (every rank: T=%d valid tokens, max S=%d; own ids / features / masks), "
                                   "train mode dropout 0.1"
                                   % (CF["label"], CF["arch_name"], NL,
                                      "MLM head (15% text masked)" if tasks == ("mlm",) else
                                      "pre-training heads, one task per step cycled " + " -> ".join(tasks) +
                                      " (15% tokens / regions masked, 1601 region labels, OT off)",
                                      CF["B"], sum(lens0), max(lens0)),
                       "global_batch": CF["B"] * world, "parallelism": "dp%d" % world,
                       "l2": "per-step working set (weights 0.22 GB + saved activations ~1 GB) exceeds the "
                             "126 MB L2; no explicit flush"},
            "e2e": {"value": round(e2e_value, 1), "unit": "samples/s", "ms_per_step": round(ms_e2e, 4),
                    "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "host_ms_per_step": round(e2e_host_ms, 3),
                    "batches": "%d distinct pinned host batches in rotation (same length profile as the "
                               "resident batch, T = %d; different ids / features / masks)"
                               % (n_host, sum(lens0))},
            "step_mode": ("eager (Python enqueues every launch)" if graphed is None else
                          "cuda_graph: fwd+bwd%s replayed per token bucket of %d (%d graphs captured, "
                          "dummy-sequence padding)" % (" + gradient all-reduce" if ar_mode == "in-graph" else
                                                       (" + gradient exchange (NVLink peer-memory kernels "
                                                        "overlapping the backward, no NCCL)" if ar_mode == "peer" else
                                                       (", all-reduce after each replay" if ar_mode == "after" else
                                                        (", one graph per layer group with the previous group's "
                                                         "all-reduce overlapped" if ar_mode == "split" else ""))),
                                                       args.token_bucket, graphed.captures)),
            "gpu_launches": int(launches), "host_enqueue_ms_per_step": round(cpu_enqueue_ms, 3),
            "algorithmic_tflops_per_step": round(flops_step / 1e12, 4),
            "achieved_tflops": round(flops_step / (ms_step * 1e-3) / 1e12, 1),
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "train_step": train_step,
            "breakdown": breakdown,
        }
        if world > 1:
            line["gradient_exchange"] = {
                "mode": ar_mode,
                "transport": ("copy-engine transfers (memcpy nodes) + ub::peer_sync_kernel / ub::peer_reduce_local_kernel "
                              "over cudaIpc-mapped NVLink peer memory (csrc/peer.cu)" if args.peer_ctas < 0 else
                              "ub::peer_push_kernel / peer_reduce_kernel / peer_allreduce_kernel over cudaIpc-mapped "
                              "NVLink peer memory (csrc/peer.cu)") if ar_mode == "peer"
                             else "ncclAllReduce(AVG) on slices of the gradient arena",
                "bytes_per_rank_per_step": int(GradArena.attach(model).numel) * 2,
                "note": peer_note}
            if peer_err:
                line["invalid"] = "a flag wait of the peer exchange expired: the gradients of this run are not reduced"
        print(json.dumps(line), file=real_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
