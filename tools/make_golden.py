#!/usr/bin/env python3
"""Regenerate ``tests/golden/``: what the unmodified reference computes in the comparisons the test-suite makes.

    python tools/make_golden.py            # the CPU runs (loss trajectory, Uni-Mol plug-in, checkpoint interchange)
    python tools/make_golden.py --gpu      # also the BERT-base fp16 loss curve on cuda:0

Needs the reference installed under ``baseline/_ref`` (see ``baseline/README.md``); the tests themselves only read the
files written here.  Every run starts from the seeded initial weights that either implementation creates by itself
(the two create identical ``state_dict`` s), so a test can regenerate its side of the comparison alone.

``reference_runs.json`` holds the logged losses, the reference's checkpoint record and what the reference reports when
it loads a checkpoint written by this framework.  ``interop_reference_checkpoint.pt`` is the reference's checkpoint with
every tensor of more than one element replaced by ``["tensor", shape, dtype, sum of |x|, max |x|, positions, values]``
(the flattened tensor's values at up to 64 seeded positions, so that a reordered layout shows): its schema, metadata
(args, optimizer history, iterator and meter state) and a fingerprint of every tensor in under 100 KB instead of the
1.8 MB of weights and moments.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden")
PY = sys.executable


def record(tool, *argv):
    out = subprocess.run([PY, os.path.join(REPO, "tools", tool)] + list(argv), env=dict(os.environ, OMP_NUM_THREADS="1"),
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800)
    if out.returncode != 0:
        raise SystemExit(out.stdout[-3000:])
    rec = json.loads([line for line in out.stdout.splitlines() if line.startswith("{")][-1])
    if "unavailable" in rec:
        raise SystemExit("{}: {}".format(tool, rec["unavailable"]))
    return rec


SAMPLES_PER_TENSOR = 64


def skeleton(obj):
    import numpy as np
    import torch

    if torch.is_tensor(obj) and obj.numel() > 1:
        flat = obj.detach().reshape(-1).float()
        n = min(SAMPLES_PER_TENSOR, flat.numel())
        idx = torch.from_numpy(np.sort(np.random.RandomState(0).choice(flat.numel(), n, replace=False)).astype(np.int32))
        return ["tensor", list(obj.shape), str(obj.dtype), float(obj.double().abs().sum()), float(flat.abs().max()),
                idx, flat[idx].clone()]
    if isinstance(obj, dict):
        return type(obj)((k, skeleton(v)) for k, v in obj.items())
    if isinstance(obj, (list, tuple)):
        return type(obj)(skeleton(v) for v in obj)
    return obj


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpu", action="store_true")
    a = ap.parse_args()
    import torch

    path = os.path.join(GOLDEN, "reference_runs.json")
    runs = json.load(open(path)) if os.path.exists(path) else {}
    with tempfile.TemporaryDirectory() as tmp:
        init = lambda name: os.path.join(tmp, name)  # noqa: E731  a fresh path: the arm creates its seeded weights
        runs["loss_parity_cpu"] = record("loss_parity.py", "--impl", "reference", "--init", init("lp.pt"), "--steps", "6")
        runs["unimol_portable_cpu"] = record("unimol_portable_check.py", "--impl", "reference", "--init", init("u.pt"),
                                             "--steps", "3")
        ref_ck, ours_ck = os.path.join(tmp, "reference.pt"), os.path.join(tmp, "ours.pt")
        runs["interop_reference"] = record("checkpoint_interop.py", "--impl", "reference", "--init", init("ci.pt"),
                                           "--steps", "3", "--save", ref_ck, "--more", "2")
        record("checkpoint_interop.py", "--impl", "ours", "--init", init("ci.pt"), "--steps", "3", "--save", ours_ck,
               "--more", "2")
        runs["interop_reference_loads_ours"] = record("checkpoint_interop.py", "--impl", "reference", "--init",
                                                      init("ci.pt"), "--load", ours_ck, "--more", "2")
        ck = torch.load(ref_ck, map_location="cpu", weights_only=False)
        torch.save(skeleton(ck), os.path.join(GOLDEN, "interop_reference_checkpoint.pt"))
        if a.gpu:
            runs["loss_curve_gpu"] = record("loss_parity.py", "--gpu", "--impl", "reference", "--init", init("g.pt"),
                                            "--steps", "12", "--dropout", "0.0", "--lr", "3e-4")
    with open(path, "w") as f:
        json.dump(runs, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", path)
    return 0


if __name__ == "__main__":
    sys.exit(main())
