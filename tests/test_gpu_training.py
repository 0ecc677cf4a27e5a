"""GPU trainer tests: fused optimizer tail, deferred (device-side) overflow handling, lazy logging output."""
import importlib
import math
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _trainer(extra):
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    importlib.import_module("bert")
    from unicore import options, tasks
    from unicore.trainer import Trainer

    parser = options.get_training_parser()
    args = options.parse_args_and_arch(parser, input_args=[
        "--task", "synthetic_mlm", "--loss", "masked_lm", "--arch", "bert_base",
        "--encoder-layers", "2", "--encoder-embed-dim", "128", "--encoder-ffn-embed-dim", "256",
        "--encoder-attention-heads", "2", "--synthetic-vocab-size", "512", "--synthetic-seq-len", "64",
        "--max-seq-len", "64", "--optimizer", "adam", "--lr", "1e-3", "--lr-scheduler", "fixed",
        "--max-update", "100", "--batch-size", "8", "--fp16", "--clip-norm", "1.0", "--seed", "5",
        "--distributed-world-size", "1", "--no-save", "--disable-validation", "--log-format", "none",
    ] + extra)
    task = tasks.setup_task(args)
    model = task.build_model(args)
    loss = task.build_loss(args)
    trainer = Trainer(args, task, model, loss)
    trainer._total_train_steps = args.max_update
    task.load_dataset("train")
    ds = task.dataset("train")
    batches = [ds.collater([ds[k * 8 + i] for i in range(8)]) for k in range(4)]
    return trainer, batches


def _run(extra, steps):
    torch.manual_seed(0)
    trainer, batches = _trainer(extra)
    outs = []
    for i in range(steps):
        outs.append(trainer.train_step([batches[i % 4]]))
    trainer.optimizer.resolve_pending_overflow()
    torch.cuda.synchronize()
    return trainer, outs


def test_deferred_overflow_matches_synchronous_path_without_overflow():
    """No overflow: identical parameters and update counts; the logging output is lazy but complete."""
    ta, outs_a = _run(["--fp16-init-scale", "4"], 6)
    tb, outs_b = _run(["--fp16-init-scale", "4", "--deferred-overflow-check"], 6)
    assert ta.get_num_updates() == tb.get_num_updates() == 6
    pa = torch.cat([p.detach().float().reshape(-1) for p in ta.model.parameters()])
    pb = torch.cat([p.detach().float().reshape(-1) for p in tb.model.parameters()])
    assert torch.isfinite(pb).all()
    assert (pa - pb).abs().max().item() < 2e-3
    la, lb = float(outs_a[-1]["loss"]), float(outs_b[-1]["loss"])
    assert math.isfinite(lb) and abs(la - lb) < 5e-2 * max(1.0, abs(la))
    assert "loss" in outs_b[-1] and "sample_size" in outs_b[-1] and len(outs_b[-1]) >= 2


def test_deferred_overflow_skips_on_device_and_rescales():
    """A loss scale far too large overflows fp16 gradients: the fused Adam kernel must leave the weights
    untouched, the scaler must come down, and skipped updates must not be counted."""
    trainer, batches = _trainer(["--fp16-init-scale", str(2 ** 24), "--deferred-overflow-check",
                                 "--fp16-scale-window", "1000"])
    before = torch.cat([p.detach().float().reshape(-1).clone() for p in trainer.model.parameters()])
    events = []
    trainer.optimizer.add_late_overflow_handler(lambda msg: events.append(msg))
    trainer.train_step([batches[0]])
    torch.cuda.synchronize()
    after = torch.cat([p.detach().float().reshape(-1) for p in trainer.model.parameters()])
    assert torch.equal(before, after), "an overflowed update must be skipped on the device"
    for i in range(1, 16):
        trainer.train_step([batches[i % 4]])
    trainer.optimizer.resolve_pending_overflow()
    torch.cuda.synchronize()
    assert len(events) >= 1
    assert trainer.optimizer.scaler.loss_scale < 2 ** 24
    assert trainer.get_num_updates() == 16 - len(events)
    final = torch.cat([p.detach().float().reshape(-1) for p in trainer.model.parameters()])
    assert torch.isfinite(final).all()
    assert not torch.equal(before, final), "training must proceed once the scale has come down"
    # Adam's bias-correction step count only advanced for the updates that really happened
    inner = trainer.optimizer.fp32_optimizer.optimizer
    steps = {int(st["step"]) for st in inner.state.values() if "step" in st}
    assert steps == {trainer.get_num_updates()}


def _gradients_after_backward(extra, micro_batches):
    """Flat gradient arena(s) after forward + backward of ``micro_batches`` (no optimizer step), dropout off."""
    torch.manual_seed(0)
    trainer, batches = _trainer(["--fp16-init-scale", "4", "--dropout", "0.0", "--attention-dropout", "0.0",
                                 "--emb-dropout", "0.0", "--activation-dropout", "0.0"] + extra)
    trainer.zero_grad()
    trainer.model.train()
    for i in range(micro_batches):
        from unicore import utils

        sample = utils.move_to_cuda(batches[i])
        trainer.task.train_step(sample, trainer.model, trainer.loss, trainer.optimizer, 0)
    torch.cuda.synchronize()
    flats = [f.grad.detach().float().clone() for g in trainer.optimizer.fp16_params for f in g["params"]]
    sinks = sum(1 for p in trainer.get_model().parameters() if getattr(p, "_ub_direct_grad", False))
    return flats, sinks


@pytest.mark.parametrize("micro_batches", [1, 3])
def test_gradient_sinks_leave_the_same_gradients_as_autograd_accumulation(micro_batches):
    """Backward kernels that add weight / bias / LayerNorm gradients straight into the flat arena
    (``ops/grad_sink.py``) against plain autograd accumulation: same arena contents, also across gradient
    accumulation micro-batches (the sink adds in fp32 before the single rounding, autograd rounds twice)."""
    direct, n_direct = _gradients_after_backward([], micro_batches)
    plain, n_plain = _gradients_after_backward(["--no-grad-sinks"], micro_batches)
    assert n_direct > 0 and n_plain == 0
    for a, b in zip(direct, plain):
        assert a.shape == b.shape and torch.isfinite(a).all()
        scale = b.abs().max().item() + 1e-12
        assert (a - b).abs().max().item() / scale < 4e-3
        assert b.abs().sum().item() > 0


def test_gradient_sinks_remove_the_accumulate_kernels():
    """The point of the sinks: far fewer ``add`` kernel launches per step (one AccumulateGrad add per parameter
    before; only the parameters outside our layer kernels - embeddings, tied LM head - afterwards)."""
    from torch.profiler import ProfilerActivity, profile

    counts = {}
    for name, extra in (("direct", []), ("plain", ["--no-grad-sinks"])):
        torch.manual_seed(0)
        trainer, batches = _trainer(["--fp16-init-scale", "4", "--deferred-overflow-check"] + extra)
        for i in range(3):
            trainer.train_step([batches[i % 4]])
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            trainer.train_step([batches[3]])
            torch.cuda.synchronize()
        counts[name] = sum(e.count for e in prof.key_averages() if "CUDAFunctor_add" in e.key)
    assert counts["direct"] < counts["plain"] - 10, counts


@pytest.mark.gpu
def test_loss_curve_tracks_the_reference_arm(tmp_path):
    """Full BERT-base (fp16, batch 32 x 512, dropout off) on this GPU, same seeded initial weights and batches: the
    logged loss of 12 updates under this framework (tcgen05 attention, fused norms, fused optimizer) and under the
    unmodified reference on a B200 (stored in ``tests/golden/reference_runs.json``) must agree to the logged precision.
    The 100-step curves are kept in profiles/loss_curve_bert_base_*."""
    import json
    import subprocess

    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(repo, "tests", "golden", "reference_runs.json")) as f:
        ref = json.load(f)["loss_curve_gpu"]["losses"]
    out = subprocess.run(
        [sys.executable, os.path.join(repo, "tools", "loss_parity.py"), "--gpu", "--impl", "ours",
         "--init", str(tmp_path / "init.pt"), "--steps", "12", "--dropout", "0.0", "--lr", "3e-4"],
        capture_output=True, text=True, timeout=600, cwd=repo)
    assert out.returncode == 0, out.stderr[-2000:]
    ours = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])["losses"]
    assert len(ours) == len(ref) == 12
    assert all(v is not None for v in ours + ref), (ours, ref)
    assert ours[-1] < ours[0] - 0.5, ours          # it trains
    assert max(abs(a - b) for a, b in zip(ours, ref)) < 0.02, (ours, ref)


@pytest.mark.gpu
def test_reading_the_loss_does_not_wait_for_the_rest_of_the_update():
    """Single process: the loss statistics are staged to the host behind the forward pass, so ``out["loss"]`` is
    answered from host numbers without materialising the device-resident meters (gradient norm ...), and it is the
    value the full materialisation reports."""
    trainer, outs = _run(["--deferred-overflow-check"], 3)
    out = outs[-1]
    assert out._values is None                      # nothing has been brought to the host on demand yet
    loss = out["loss"]
    assert isinstance(loss, float) and out._values is None
    assert "loss" in out and "no_such_key" not in out and out.get("no_such_key", 7) == 7
    everything = dict(out.items())                  # full materialisation (one host transfer for what is left)
    assert everything["loss"] == loss and "seq_len" in everything and "sample_size" in everything
