"""Trained acting nets for the tests: snapshots of the engine's own training (SelfPlay + Learner).

    python oracle/gen_trained_nets.py [--out tests/golden/trained_nets.npz] [--seed 1234] [--commit HASH]

Freshly initialised nets give outputs near 1; trained ones do not: a best-response net predicts returns of several chips
and an average policy is close to deterministic in many states.  tests/act_reference.py loads these snapshots as its
"trained-*" families.  One SGD run at config.ini's rates is saved at three points and one Adam run at one point, all at
65 536 games and rollout(8) + Learner.update() per iteration (main.train's loop).  The file records the command, seed,
iterations, commit, card name and power limit.  Needs a GPU."""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GAMES = 65536
SNAPSHOTS = (("sgd", (5000, 20000, 60000)), ("adam", (20000,)))


def _commit(given):
    if given:
        return given
    r = subprocess.run(["git", "rev-parse", "HEAD"], cwd=ROOT, capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown"


def train(optimizer, points, seed):
    import torch

    import nfsp_b200
    from nfsp_b200.learner import Learner

    sp = nfsp_b200.SelfPlay(GAMES, seed=seed, max_steps_per_call=8, direct_rings="auto")
    ln = Learner(sp, optimizer=optimizer)
    out, it = [], 0
    for stop in points:
        while it < stop:
            sp.rollout(8)
            ln.update(sync=False)
            it += 1
        torch.cuda.synchronize()
        out.append((it, sp.weights.cpu().numpy().copy()))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "trained_nets.npz"))
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--commit", default="", help="commit of the training code (default: git rev-parse HEAD)")
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()[0].split(", ")
    labels, ws, iters, opts = [], [], [], []
    t0 = time.time()
    for opt, points in SNAPSHOTS:
        for it, w in train(opt, points, a.seed):
            labels.append("%s-%d" % (opt, it))
            ws.append(w)
            iters.append(it)
            opts.append(opt)
    seconds = time.time() - t0
    from nfsp_b200 import exploitability as ex

    obs = np.array(sorted(set(ex.information_states()[0]) | set(ex.information_states()[1])), np.int64)
    x = ((obs[:, None] >> np.arange(30)) & 1).astype(np.float64)
    report = []
    for label, w in zip(labels, ws):
        qmax, span = 0.0, 0.0
        for k in range(4):
            v = w[k].astype(np.float64)
            z = np.maximum(x @ v[:1920].reshape(30, 64) + v[1920:1984], 0) @ v[1984:2176].reshape(64, 3) + v[2176:]
            span = max(span, float((z.max(1) - z.min(1)).max()))
            if k & 1:
                qmax = max(qmax, float(np.abs(z).max()))
        report.append("%s: max |Q| %.2f chips, largest logit span %.2f" % (label, qmax, span))
        assert qmax >= 1.0, "snapshot %s has no Q-value of a chip: train longer" % label
    np.savez_compressed(a.out, labels=np.array(labels), w=np.stack(ws).astype(np.float32), iterations=np.array(iters),
                        optimizer=np.array(opts), seed=np.int64(a.seed), games=np.int64(GAMES),
                        command=np.array("python oracle/gen_trained_nets.py --seed %d" % a.seed),
                        commit=np.array(_commit(a.commit)), card=np.array(card[0]),
                        power_limit=np.array(card[1] if len(card) > 1 else "unknown"),
                        train_seconds=np.float64(seconds))
    print("card %s, power limit %s; %.1f s of training" % (card[0], card[1] if len(card) > 1 else "?", seconds))
    print("\n".join(report))


if __name__ == "__main__":
    main()
