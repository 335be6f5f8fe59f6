"""The float64 reference of the learner's fit (oracle/learner_oracle.fit) against torch.autograd and plain float64 SGD
steps on the CPU.  The loss is defined as in test_gpu_learner.test_gradients_match_torch_autograd: Dense-relu-Dense;
a relu head with the Huber loss of agent.py:91-99 averaged over the three outputs, or a softmax head with categorical
cross-entropy on the target as given.  Autograd derives the backward pass from that definition, so the reference the
GPU tests hold the kernels to shares nothing with the hand-written backward passes.  No GPU needed."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import learner_oracle as lo  # noqa: E402


def _autograd_fit(c, minibatch, fit_batch, epochs, gamma, mask, terminal_bootstraps, others_to_target):
    """Keras' fit() restated with torch: the batches of `fit_batch` rows of every epoch (the last one ragged), one
    float64 SGD step each.  Returns the weights and the first step's statistics (layout of lo.fit)."""
    import torch.nn.functional as F

    def parts(w):
        return w[:1920].reshape(30, 64), w[1920:1984], w[1984:2176].reshape(64, 3), w[2176:2179]

    def net(w, m):
        W1, b1, W2, b2 = parts(w)
        x = torch.from_numpy(((np.asarray(m, np.uint32)[:, None] >> np.arange(30)) & 1).astype(np.float64))
        return F.relu(x @ W1 + b1) @ W2 + b2

    W = [torch.from_numpy(c["w"][k].copy()) for k in range(4)]
    T = [torch.from_numpy(c["w_target"][p].copy()) for p in range(2)]
    stats = [float("nan")] * 8
    for epoch in range(epochs):
        for step, rows in enumerate(torch.arange(minibatch).split(fit_batch)):
            rows = rows.numpy()
            for k in range(4):
                if not (mask >> k) & 1:
                    continue
                p, w = k >> 1, W[k].clone().requires_grad_(True)
                if k & 1:
                    b = c["rl"][p][rows]
                    q = F.relu(net(w, b["s"]))
                    with torch.no_grad():
                        qs = F.relu(net(T[p], b["s"]))
                        live = 1.0 if terminal_bootstraps else 1.0 - torch.from_numpy(b["t"].astype(np.float64))
                        y = torch.from_numpy(b["r"].astype(np.float64)) + gamma * live * F.relu(net(T[p], b["s2"])).max(1).values
                        tgt = qs.clone() if others_to_target else q.detach().clone()
                        tgt[torch.arange(len(rows)), torch.from_numpy(b["a"].astype(np.int64))] = y
                    err = tgt - q
                    huber = torch.where(err.abs() > 1, err.abs() - 0.5, 0.5 * err * err).mean(dim=1)
                    huber.mean().backward()
                    if epoch == 0 and step == 0:
                        stats[4 + k], stats[p], stats[2 + p] = float(huber.detach().sum()), float(qs.max(1).values.sum()), len(rows)
                else:
                    b = c["sl"][p][rows]
                    y = torch.from_numpy(b["a"].astype(np.float64))
                    z = net(w, b["s"])
                    (-(y * F.log_softmax(z, dim=1)).sum(1)).mean().backward()
                    if epoch == 0 and step == 0:   # the reported loss clamps the probabilities at 1e-7, as Keras does
                        stats[4 + k] = float(-(y * torch.log(torch.clamp(F.softmax(z.detach(), dim=1), min=1e-7))).sum())
                W[k] = (w - c["lr"][k] * w.grad).detach()
    return torch.stack(W).numpy(), np.array(stats)


@pytest.mark.parametrize("terminal_bootstraps", [False, True])
@pytest.mark.parametrize("others_to_target", [False, True])
@pytest.mark.parametrize("minibatch,fit_batch,epochs,mask", [
    (128, 32, 2, 0xF),       # the reference's sizes
    (100, 24, 3, 0xF),       # ragged last slice of 4 rows, three epochs
    (33, 8, 1, 0b0101),      # a last slice of one row; only the average-policy nets train
    (70, 64, 2, 0b1010),     # only the best-response nets train
])
def test_fit_reference_matches_autograd_sgd(minibatch, fit_batch, epochs, mask, terminal_bootstraps, others_to_target):
    c = lo.fit_case(3, minibatch)
    w, stats, margin, seen = lo.fit(c["w"], c["w_target"], c["rl"], c["sl"], minibatch, fit_batch, epochs, c["lr"], 0.95,
                                    mask, terminal_bootstraps, others_to_target)
    w_ref, stats_ref = _autograd_fit(c, minibatch, fit_batch, epochs, 0.95, mask, terminal_bootstraps, others_to_target)
    assert np.abs(w - w_ref).max() <= 1e-12
    assert np.array_equal(np.isnan(stats), np.isnan(stats_ref))
    ok = ~np.isnan(stats)
    assert np.allclose(stats[ok], stats_ref[ok], rtol=1e-12, atol=1e-12), (stats, stats_ref)
    for k in range(4):
        if (mask >> k) & 1:
            assert np.abs(w[k] - c["w"][k]).max() > 1e-3          # every trained net moved
        else:
            assert np.array_equal(w[k], c["w"][k])                 # the others are untouched
    assert margin > 0
    if mask & 0b1010:
        assert seen["huber_linear"] > 0 and seen["huber_quadratic"] > 0
    if mask & 0b0100:
        assert seen["log_clamped"] > 0


def test_fit_case_has_its_edges():
    """The hand-built records carry every edge the GPU tests rely on, and the SL targets include unnormalised and
    all-zero ones."""
    c = lo.fit_case(0, 128)
    for p in range(2):
        rl, sl = c["rl_slots"][p], c["sl_slots"][p]
        for m in (rl["s"], rl["s2"], sl["s"]):
            assert 0 in m and 0x3FFFFFFF in m
        assert set(np.unique(rl["t"])) == {0, 1} and rl["r"].min() < -12 and rl["r"].max() > 12
        ysum = sl["a"].sum(1)
        assert (ysum == 0).any() and (ysum == 1).any() and ((ysum != 0) & (ysum != 1)).any()
        for idx in (c["idx_rl"][p], c["idx_sl"][p]):
            assert len(np.unique(idx)) < len(idx) and (np.diff(idx) < 0).any()
        for m in (c["rl"][p]["s"], c["rl"][p]["s2"], c["sl"][p]["s"]):   # the sampled rows hold the edges too
            assert 0 in m and 0x3FFFFFFF in m
        assert (c["sl"][p]["a"].sum(1) == 0).any()
    z = np.maximum(lo.bits(c["sl"][1]["s"]) @ lo.split(c["w"][2])[0] + lo.split(c["w"][2])[1], 0) @ lo.split(c["w"][2])[2] \
        + lo.split(c["w"][2])[3]
    assert (z.max(1) - z.min(1)).min() > 100                       # player 1's average net: logits span > 100
    assert len(set(c["lr"].tolist())) == 4
