#!/usr/bin/env python3
"""Headline benchmark: BERT-base masked-LM training throughput (samples/s, whole job).

``python bench.py --gpus N --steps K --warmup W`` (for N>1 the same command under
``torch.distributed.run``): W untimed steps, then exactly K steps timed on the device with CUDA events
between barrier+synchronize pairs, MAX over ranks, one JSON line from rank 0.  Weights, batches and
dropout are seeded, so the same arguments give the same inputs on every run; ``--dump-outputs DIR``
writes what the last timed step returned (see ``dump_outputs``) to compare two builds output for output.

Metric/config = BASELINE.json config 2 / BASELINE.md B1: ``bert_base`` (12L-768-3072-12H, vocab
30,522, rel-pos bias), fp16 with dynamic loss scaling, Adam(0.9, 0.98, eps 1e-6), clip-norm 1.0,
polynomial-decay LR, sequence length 512, synthetic tokens (15 % masked), random-init weights,
per-GPU batch fixed (weak scaling).  A step = forward + backward + gradient reduction + clip +
optimizer update + stats, i.e. one ``Trainer.train_step`` - nothing is skipped.

``--impl reference`` runs the UNMODIFIED reference installed in ``baseline/_ref`` (pure-PyTorch
fallback ops, torch DDP/NCCL) through the same harness: its own ``Trainer.train_step`` on its own
``examples/bert`` model, same batches, same flags.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading

REPO = os.path.dirname(os.path.abspath(__file__))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--arch", default="bert_base")
    ap.add_argument("--batch-size", type=int, default=32, help="sentences per GPU per step")
    ap.add_argument("--seq-len", type=int, default=512)
    ap.add_argument("--vocab", type=int, default=30522)
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--update-freq", type=int, default=1)
    ap.add_argument("--ema-decay", type=float, default=-1.0)
    ap.add_argument("--ddp-backend", default=None)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--ref-ext", action="store_true",
                    help="reference arm only: make the reference's OWN CUDA extensions importable (rebuilt with an sm_100 "
                         "gencode into baseline/_ref_ext by baseline/build_ref_ext.sh) = BASELINE.md B2; the default "
                         "reference arm is its stock install without extensions (B1)")
    ap.add_argument("--report-losses", action="store_true", help="add the losses read back in the end-to-end region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's logging output and a seeded sample of the "
                         "updated weights to DIR/<name>.npy (rank 0)")
    ap.add_argument("--sync-overflow-check", action="store_true",
                    help="ours: read the grad norm on the host every step (reference behaviour) instead of the "
                         "deferred, device-side overflow skip")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    FIELDS = (
        "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
        "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    )

    def __init__(self, device_index=0):
        self.device_index = device_index
        self.proc = None
        self.lines = []
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.device_index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
        except Exception:  # noqa: BLE001
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.lines.append(line.strip())

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(smax) if smax else None,
            "power_w_max": max(power) if power else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


# ------------------------------------------------------------------------------------------------
# harness pieces shared by both arms (they only use the public unicore API)
# ------------------------------------------------------------------------------------------------
def make_batches(n, bsz, seq_len, vocab, pad_idx, mask_idx, special, seed):
    """n CPU batches of the masked-LM contract; 15 % of positions masked, no padding."""
    import numpy as np
    import torch

    rng = np.random.RandomState(seed)
    allowed = np.setdiff1d(np.arange(vocab), np.asarray(sorted(special)))
    n_mask = max(1, int(round(0.15 * seq_len)))
    out = []
    for _ in range(n):
        tokens = allowed[rng.randint(0, len(allowed), size=(bsz, seq_len))]
        target = np.full((bsz, seq_len), pad_idx, dtype=np.int64)
        src = tokens.copy()
        for b in range(bsz):
            pos = rng.choice(seq_len, n_mask, replace=False)
            target[b, pos] = tokens[b, pos]
            src[b, pos] = mask_idx
        out.append({
            "net_input": {"src_tokens": torch.from_numpy(src.astype(np.int64))},
            "target": torch.from_numpy(target),
        })
    return out


def train_flags(a, world):
    flags = [
        "--task", "bench_mlm", "--loss", "masked_lm", "--arch", a.arch,
        "--optimizer", "adam", "--adam-betas", "(0.9, 0.98)", "--adam-eps", "1e-6", "--clip-norm", "1.0",
        "--lr-scheduler", "polynomial_decay", "--lr", "1e-4", "--warmup-updates", "100",
        "--total-num-update", "10000", "--max-update", "10000",
        "--batch-size", str(a.batch_size), "--update-freq", str(a.update_freq), "--seed", "1",
        "--num-workers", "0", "--log-format", "none", "--disable-validation", "--no-save",
        "--max-seq-len", str(max(512, a.seq_len)),
        "--distributed-world-size", str(world),
    ]
    if a.precision == "fp16":
        flags += ["--fp16", "--fp16-init-scale", "4", "--fp16-scale-window", "256"]
        if getattr(a, "impl", "ours") != "reference" and not getattr(a, "sync_overflow_check", False):
            flags += ["--deferred-overflow-check"]  # ours only: see unicore/options.py
    else:
        flags += ["--bf16"]
    if a.ema_decay > 0:
        flags += ["--ema-decay", str(a.ema_decay)]
    return flags


def setup_paths(impl, ref_ext=False):
    if impl == "reference":
        ref = os.path.join(REPO, "baseline", "_ref")
        if not os.path.isdir(os.path.join(ref, "unicore")):
            return "baseline/_ref/unicore not found (reference not installed)"
        if not os.path.isfile(os.path.join(ref, "examples", "bert", "model.py")):
            return "baseline/_ref/examples/bert not found (reference example model missing)"
        # reference first, then its examples (so `import bert` finds the reference model), then stubs
        for p in (os.path.join(REPO, "baseline", "stubs"), os.path.join(ref, "examples"), ref):
            sys.path.insert(0, p)
        if ref_ext:
            ext = os.path.join(REPO, "baseline", "_ref_ext")
            if not any(f.startswith("unicore_fused_layernorm") for f in (os.listdir(ext) if os.path.isdir(ext) else [])):
                return "baseline/_ref_ext has no rebuilt reference extensions (run baseline/build_ref_ext.sh)"
            sys.path.insert(0, ext)
        # make sure OUR packages are not importable on this arm
        sys.path[:] = [p for p in sys.path if os.path.abspath(p or ".") != REPO]
        for mod in list(sys.modules):
            if mod == "unicore" or mod.startswith("unicore.") or mod.startswith("unicore_b200"):
                del sys.modules[mod]
    else:
        if REPO not in sys.path:
            sys.path.insert(0, REPO)
    return None


def register_bench_task(impl):
    """A task named ``bench_mlm`` that only provides the dictionary (batches come from make_batches)."""
    from unicore.data import Dictionary
    from unicore.tasks import UnicoreTask, register_task, TASK_REGISTRY

    if "bench_mlm" in TASK_REGISTRY:
        return

    @register_task("bench_mlm")
    class BenchMLMTask(UnicoreTask):
        @staticmethod
        def add_args(parser):
            parser.add_argument("--bench-vocab", type=int, default=30522)

        def __init__(self, args, dictionary):
            super().__init__(args)
            self.dictionary = dictionary
            self.mask_idx = dictionary.add_symbol("[MASK]", is_special=True)

        @classmethod
        def setup_task(cls, args, **kwargs):
            specials = {0: "[PAD]", 100: "[UNK]", 101: "[CLS]", 102: "[SEP]", 103: "[MASK]"}
            d = Dictionary()
            for i in range(args.bench_vocab):
                d.add_symbol(specials.get(i, "t{}".format(i)))
            return cls(args, d)

        def load_dataset(self, split, **kwargs):
            raise RuntimeError("bench task has no datasets")


def build_trainer(a, impl, world, rank, local_rank):
    import torch

    if impl == "reference":
        import bert  # noqa: F401  reference examples/bert: registers model "bert" + its task
    else:
        import importlib

        sys.path.insert(0, os.path.join(REPO, "examples"))
        importlib.import_module("bert")  # our plug-in (examples/bert)
    from unicore import options, tasks
    from unicore.trainer import Trainer

    register_bench_task(impl)
    parser = options.get_training_parser()
    flags = train_flags(a, world) + ["--bench-vocab", str(a.vocab)]
    # ours: gradient all-reduce on the hand-written NVLink peer-memory kernels (falls back to c10d with a
    # warning when symmetric memory is unavailable); reference: its own default (c10d DDP)
    backend = a.ddp_backend or ("b200" if (impl != "reference" and world > 1) else "c10d")
    flags += ["--ddp-backend", backend, "--device-id", str(local_rank), "--distributed-rank", str(rank)]
    args = options.parse_args_and_arch(parser, input_args=flags)
    args.distributed_rank = rank
    args.device_id = local_rank
    torch.manual_seed(args.seed)  # the initial weights
    task = tasks.setup_task(args)
    model = task.build_model(args)
    loss = task.build_loss(args)
    trainer = Trainer(args, task, model, loss)
    trainer._total_train_steps = args.max_update  # what init_total_train_steps() would set
    return args, task, trainer


DUMP_PARAM_SAMPLE = 1 << 22  # 16 MB of float32
TIMING_STATS = ("wall", "train_wall", "ups", "gb_free")  # differ from run to run by nature


def dump_outputs(out_dir, stats, model):
    """What a caller of ``Trainer.train_step`` receives from the step: its logging output (one float64 array per
    numeric statistic, timing meters left out) and the updated model, as ``params_sample.npy``: float32 values at
    2^22 positions of all parameters flattened in ``named_parameters()`` order, drawn (with replacement) from a fixed
    seed."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name, value in stats.items():
        if name in TIMING_STATS:
            continue
        arr = np.asarray(value.detach().cpu().double().numpy() if torch.is_tensor(value) else value)
        if arr.dtype.kind in "biuf":
            np.save(os.path.join(out_dir, name + ".npy"), arr.astype(np.float64))
    with torch.no_grad():
        flat = torch.cat([p.detach().reshape(-1).float() for _, p in model.named_parameters()])
        idx = torch.from_numpy(np.sort(np.random.RandomState(0).randint(0, flat.numel(), size=DUMP_PARAM_SAMPLE)))
        np.save(os.path.join(out_dir, "params_sample.npy"), flat[idx.to(flat.device)].cpu().numpy())


def count_launches_start(impl):
    if impl != "ours":
        return None
    from unicore_b200.ops import _native

    return _native.launch_counter_reset()


def count_launches_stop(impl):
    if impl != "ours":
        return None
    from unicore_b200.ops import _native

    return _native.launch_counter_read()


def main():
    a = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        a.gpus = world

    why = setup_paths(a.impl, a.ref_ext)
    if why is not None:
        if rank == 0:
            print(json.dumps({"impl": a.impl, "unavailable": why}))
        return 0

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        if rank == 0:
            print(json.dumps({"impl": a.impl, "unavailable": "no CUDA device visible"}))
        return 0
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend="nccl", init_method="env://", world_size=world, rank=rank)
        dist.all_reduce(torch.zeros(1, device="cuda"))

    try:
        args, task, trainer = build_trainer(a, a.impl, world, rank, local_rank)
    except Exception as exc:  # noqa: BLE001
        if a.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "reference failed to build: {!r}".format(exc)[:300]}))
            return 0
        raise

    d = task.dictionary
    n_distinct = 8
    cpu_batches = make_batches(
        n_distinct, a.batch_size * a.update_freq, a.seq_len, len(d), d.pad(), task.mask_idx,
        special=[d.pad(), d.unk(), d.bos(), d.eos(), task.mask_idx], seed=1234 + rank,
    )

    def split_micro(batch):
        if a.update_freq == 1:
            return [batch]
        out = []
        for i in range(a.update_freq):
            sl = slice(i * a.batch_size, (i + 1) * a.batch_size)
            out.append({"net_input": {"src_tokens": batch["net_input"]["src_tokens"][sl]}, "target": batch["target"][sl]})
        return out

    pinned = [{"net_input": {"src_tokens": b["net_input"]["src_tokens"].pin_memory()}, "target": b["target"].pin_memory()}
              for b in cpu_batches]
    on_device = [{"net_input": {"src_tokens": b["net_input"]["src_tokens"].cuda()}, "target": b["target"].cuda()}
                 for b in cpu_batches]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    seen_losses = []

    def run_steps(batches, n, read_loss):
        out = None
        for i in range(n):
            out = trainer.train_step(split_micro(batches[i % len(batches)]))
            if read_loss and out is not None:
                v = out.get("loss", None)
                seen_losses.append(float(v) if v is not None else None)  # device -> host read of the step result
        return out

    # ---- warm-up (builds optimizer, allocator high-water mark, cuBLAS heuristics, loss scale) ----
    run_steps(on_device, max(3, a.warmup), read_loss=False)
    barrier()

    # ---- timed region 1: device-resident inputs, CUDA events ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    count_launches_start(a.impl)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    last_out = run_steps(on_device, a.steps, read_loss=False)
    stop.record()
    barrier()
    launches = count_launches_stop(a.impl)
    elapsed_ms = start.elapsed_time(stop)
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        if last_out is None:
            raise RuntimeError("the last timed step returned no logging output (an fp16 overflow skipped it)")
        dump_outputs(a.dump_outputs, last_out, trainer.get_model())
    t = torch.tensor([elapsed_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())

    # ---- timed region 2: end to end (pinned host batch -> H2D each step, loss read back each step) ----
    e2e = None
    if not a.no_e2e:
        barrier()
        s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s2.record()
        run_steps(pinned, a.steps, read_loss=True)
        e2.record()
        barrier()
        t2 = torch.tensor([s2.elapsed_time(e2)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        e2e_ms = float(t2.item())
        h2d = sum(x.numel() * x.element_size() for x in (pinned[0]["net_input"]["src_tokens"], pinned[0]["target"]))
        e2e = {
            "value": world * a.batch_size * a.update_freq * a.steps / (e2e_ms / 1e3),
            "unit": "samples/s",
            "ms_per_step": e2e_ms / a.steps,
            "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": 8,
        }

    if rank == 0:
        global_batch = world * a.batch_size * a.update_freq
        value = global_batch * a.steps / (elapsed_ms / 1e3)
        result = {
            "metric": "{} masked-LM training throughput (samples/s, whole job, device-timed, max over ranks)".format(
                {"bert_base": "BERT-base", "bert_large": "BERT-large"}.get(a.arch, a.arch)),
            "impl": a.impl,
            "reference_cuda_ext": bool(a.ref_ext) if a.impl == "reference" else None,
            "value": value,
            "unit": "samples/s",
            "n_gpus": world,
            "steps": a.steps,
            "warmup": max(3, a.warmup),
            "ms_per_step": elapsed_ms / a.steps,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,  # BASELINE.md publishes no number; the driver compares against --impl reference
            "dtype": a.precision,
            "data": "synthetic tokens (15% masked, no padding), random-init weights",
            "tokens_per_s": value * a.seq_len,
            "config": {
                "model": a.arch,
                "global_batch": global_batch,
                "per_gpu_batch": a.batch_size,
                "update_freq": a.update_freq,
                "seq_len": a.seq_len,
                "vocab": a.vocab,
                "parallelism": "dp{}".format(world),
                "ddp_backend": getattr(args, "ddp_backend", None),
                "optimizer": "adam(0.9,0.98) clip 1.0 polynomial_decay, {}".format(
                    "fp16 dynamic loss scale" if a.precision == "fp16" else "bf16 (no loss scaling)"),
                "overflow_check": "host read every step (reference behaviour)"
                if (a.impl == "reference" or a.precision != "fp16" or a.sync_overflow_check)
                else "decided on the device; the loss scaler is told before the next backward",
                "optimizer_tail": "fused (one kernel after backward)"
                if getattr(getattr(trainer, "optimizer", None), "uses_fused_tail", False) else "replicated",
                "ema_decay": a.ema_decay if a.ema_decay > 0 else None,
                "l2": "no explicit flush: each step streams >1.7 GB of weights/optimizer state/activations, "
                      "far above the 126 MB L2, and 8 distinct input batches rotate",
            },
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": launches,
        }
        if a.report_losses:
            result["losses"] = seen_losses[:16]
        print(json.dumps(result))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
