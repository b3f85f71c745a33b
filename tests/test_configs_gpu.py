"""Parity at the sizes BASELINE.json's configs actually use, against golden outputs the UNMODIFIED
reference produced at those sizes (oracle/make_golden_configs.py -> tests/golden/cfg*_golden.pt,
train18_golden.pt).  Seeded torch CPU generators recreate the reference's inputs bit for bit.

Bars: permutations identical to the reference's, or — where the GPU's fp32 forward (cuDNN) and the
CPU's (oneDNN) move a near-tie — an equal optimum within 1e-6 relative on the reference's own cost
matrix (configs 1 and 2 recompute it with the oracle port, itself checked against the stored
fingerprints); cost matrices within 1e-4 of the largest entry (north-star bar);
partial_merge tensors BIT-equal (sha256) whenever the permutations are identical; PLeaS logits
after the drivers' BN reset within the tolerances written in test_train_rn18_logits_*.
"""
import hashlib
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, key_str, load_spec_json
from oracle import ref_oracle as O

pytestmark = pytest.mark.gpu
N_SAMPLES = 256


def _pkg():
    import pleas_merging_b200 as P

    return P


def _load(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def _pair(arch):
    import torchvision

    torch.manual_seed(0)
    m1 = getattr(torchvision.models, arch)().eval()
    torch.manual_seed(1)
    m2 = getattr(torchvision.models, arch)().eval()
    return m1, m2


def _loader(nb, b, hw, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(b, 3, hw, hw, generator=g), 0) for _ in range(nb)]


def _sample_index(n):  # oracle/make_golden_configs.py::sample_index
    rng = np.random.default_rng(1000 + n)
    return rng.integers(0, n, N_SAMPLES), rng.integers(0, n, N_SAMPLES)


# Largest relative deviation of a group's optimal objective from the reference's.  The forwards of the source
# models run on the library's 3xTF32 tensor-core convolution (csrc/conv.cu).  The tensor core truncates when it
# accumulates, a bias that compounds from layer to layer, so the kernel promotes two-box (64 k) chains and issues
# their small products first; measured worst deviation on the ResNet-50 pair: 4.2e-6 (one-box chains 3.2e-6,
# eight-box chains in k order 1.3e-5; cuDNN fp32 forwards ~4e-6).
OBJ_TOL = 1e-5


def _check_fingerprint(cost, fp, name, tol=1e-5):
    """cost (CUDA fp32 [n, n]) against the stored row / column sums, diagonal and sampled entries of the
    reference's matrix; errors relative to the largest entry (sums: to n times it)."""
    c = cost.detach().cpu()
    n = c.shape[0]
    scale = fp["absmax"]
    d = c.double()
    assert float((d.sum(1) - fp["rowsum"]).abs().max()) <= tol * n * scale, name
    assert float((d.sum(0) - fp["colsum"]).abs().max()) <= tol * n * scale, name
    assert float((c.diagonal() - fp["diag"]).abs().max()) <= 10 * tol * scale, name
    r, s = _sample_index(n)
    mine = c[torch.from_numpy(r), torch.from_numpy(s)]
    assert float((mine - fp["samples"]).abs().max()) <= 10 * tol * scale, name


def _relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def _perm_or_objective(perm, gold, cost, name):
    """Returns the number of differing assignments; asserts an equal optimum (1e-6 rel) when > 0."""
    perm, gold = np.asarray(perm, dtype=np.int64), np.asarray(gold, dtype=np.int64)
    flips = int((perm != gold).sum())
    if flips:
        c = np.asarray(cost, dtype=np.float64)
        idx = np.arange(len(perm))
        a, b = c[idx, perm].sum(), c[idx, gold].sum()
        assert abs(a - b) <= 1e-6 * abs(b), f"{name}: objective {a} vs reference {b} ({flips} assignments differ)"
    return flips


def _digest(t):
    t = t.detach().cpu().contiguous()
    d = t.double()
    return hashlib.sha256(t.numpy().tobytes()).hexdigest(), float(d.sum()), float((d * d).sum())


# ----------------------------------------------------------------------------------------- config 1

def test_config1_rn18_activation_matching_and_merge_vs_reference():
    """BASELINE config 1 in full: ResNet-18 pair, 10 batches of 32x3x224x224, reference semantics
    (last batch) and the accumulate-fixed sum; partial_merge at ratio 0.0."""
    P = _pkg()
    G = _load("cfg1_rn18_golden.pt")
    m1, m2 = _pair("resnet18")
    spec = P.get_permutation_spec(m1, ((1, 3, 224, 224),))
    loader = _loader(*G["loader"])
    # the reference's full cost matrices are not stored (4.2 MB): the verbatim mode depends on the last batch
    # only, so the oracle port recomputes them on the host, tied to the reference by the stored fingerprints
    ocosts = O.matching_costs(load_spec_json("resnet18"), m1, m2, loader[-1:], 1, "cdist", "reference")
    for k in spec:
        oc = torch.from_numpy(np.ascontiguousarray(ocosts[(k.key, k.axis)]))
        _check_fingerprint(oc, G["am/reference/fingerprint"][key_str(k)], "oracle " + key_str(k), tol=1e-6)
    m1, m2 = m1.cuda(), m2.cuda()
    perm, costs = P.activation_matching(spec, m1, m2, loader, num_batches=10, output_costs=True)
    flips = 0
    for k in spec:
        ks = key_str(k)
        _check_fingerprint(costs[k], G["am/reference/fingerprint"][ks], ks)
        oc = ocosts[(k.key, k.axis)]
        assert _relerr(costs[k].cpu().numpy(), oc) <= 1e-4, ks
        flips += _perm_or_objective(perm[k].numpy(), G["am/reference/perm"][ks].numpy(), oc, ks)
    print("config 1 (reference mode): assignments differing from the reference:", flips)
    assert flips == 0  # observed; the objective escape hatch above documents the contract if this ever moves
    model3 = P.partial_merge(spec, m1, m2, perm, costs, {k: 0.0 for k in spec})
    sd = model3.state_dict()
    assert set(sd) == set(G["pm/r0/digest"])
    for name, (sha, s1, s2) in G["pm/r0/digest"].items():
        assert _digest(sd[name])[0] == sha, name  # gathers and (a + b) / 2: bit exact
    # paper-intended sum over the 10 batches (oracle = reference with the one-token F1 fix)
    perm_s, costs_s = P.activation_matching(spec, m1, m2, loader, num_batches=10, output_costs=True, accumulate="sum")
    flips = 0
    for k in spec:
        ks = key_str(k)
        _check_fingerprint(costs_s[k], G["am/sum/fingerprint"][ks], ks)
        flips += _perm_or_objective(perm_s[k].numpy(), G["am/sum/perm"][ks].numpy(), costs_s[k].cpu().numpy(), ks)
        obj = float(costs_s[k].double().cpu()[torch.arange(len(perm_s[k])), perm_s[k]].sum())
        # the reference's own fp32 pipeline (SGEMM over K = 401 408, ten fp32 adds) is only good to ~2e-6
        assert abs(obj - G["am/sum/obj"][ks]) <= OBJ_TOL * abs(G["am/sum/obj"][ks]), ks
    print("config 1 (sum mode): assignments differing from the reference:", flips)


# ----------------------------------------------------------------------------------------- config 2

def test_config2_rn50_last_batch_vs_reference():
    """BASELINE config 2 in the reference's verbatim mode: only the last processed batch counts
    (SURVEY F1), so the reference's result on [batch] equals its result on [decoys..., batch].  The
    product is run on three batches (two decoys first) of 32x3x224x224 and must reproduce the
    reference's 37 permutations."""
    P = _pkg()
    G = _load("cfg2_rn50_golden.pt")
    m1, m2 = _pair("resnet50")
    spec = P.get_permutation_spec(m1, ((1, 3, 224, 224),))
    last = _loader(*G["loader"])
    loader = _loader(2, 32, 224, 77) + last
    # the reference's full cost matrices are not stored (32 MB): the oracle port recomputes them on the host
    # from the same batch and is tied to the reference by the stored fingerprints
    ocosts = O.matching_costs(load_spec_json("resnet50"), m1, m2, last, 1, "cdist", "reference")
    for k in spec:
        ks = key_str(k)
        fp = G["am/reference/fingerprint"][ks]
        oc = torch.from_numpy(np.ascontiguousarray(ocosts[(k.key, k.axis)]))
        _check_fingerprint(oc, fp, "oracle " + ks, tol=2e-6)
    perm, costs = P.activation_matching(spec, m1.cuda(), m2.cuda(), loader, num_batches=3, output_costs=True)
    flips, worst, worst_obj = 0, 0.0, 0.0
    for k in spec:
        ks = key_str(k)
        _check_fingerprint(costs[k], G["am/reference/fingerprint"][ks], ks)
        oc = ocosts[(k.key, k.axis)]
        worst = max(worst, _relerr(costs[k].cpu().numpy(), oc))
        flips += _perm_or_objective(perm[k].numpy(), G["am/reference/perm"][ks].numpy(), oc, ks)
        obj = float(costs[k].double().cpu()[torch.arange(len(perm[k])), perm[k]].sum())
        worst_obj = max(worst_obj, abs(obj - G["am/reference/obj"][ks]) / abs(G["am/reference/obj"][ks]))
    print(f"config 2: worst objective deviation from the reference {worst_obj:.2e}")
    assert worst_obj <= OBJ_TOL
    assert worst <= 1e-4
    print(f"config 2: max cost rel-err {worst:.2e}; assignments differing from the reference: {flips} of "
          f"{sum(pg.size for pg in spec.values())}")


# ----------------------------------------------------------------------------------------- config 3

def test_config3_rn50_weight_matching_and_budget_merges_vs_reference(capsys):
    """BASELINE config 3: ResNet-50 weight_matching(seed=0) — all 37 permutations identical to the
    reference's, same number of LAP solves — then partial_merge at budgets 1.2 / 1.55 / 1.8 / 2.0 with
    the drivers' zip rule: block index lists and every merged tensor bit-equal."""
    P = _pkg()
    G = _load("cfg3_rn50_golden.pt")
    m1, m2 = _pair("resnet50")
    spec = P.get_permutation_spec(m1, ((1, 3, 224, 224),))
    m1, m2 = m1.cuda(), m2.cuda()
    perm, costs = P.weight_matching(spec, m1.state_dict(), m2.state_dict(), max_iter=100, seed=0, verbose=True,
                                    return_costs=True)
    visits = [ln for ln in capsys.readouterr().out.splitlines() if "/" in ln and ":" in ln]
    assert len(visits) == G["wm/lap_calls"]  # 666 visits = 18 sweeps x 37 groups, one LAP each
    for k in spec:
        ks = key_str(k)
        assert (perm[k].numpy() == G["wm/perm"][ks].numpy().astype(np.int64)).all(), ks
        _check_fingerprint(costs[k], G["wm/fingerprint"][ks], ks)
    for budget in (1.2, 1.55, 1.8, 2.0):
        tag = f"pm/{budget}"
        ratios = {k: G[f"{tag}/ratios"][key_str(k)] for k in spec}
        model3, blocks = P.partial_merge(spec, m1, m2, perm, costs, ratios, return_blocks=True)
        for k in spec:
            ks = key_str(k)
            assert [len(t) for t in blocks[k]] == G[f"{tag}/block_sizes"][ks], (budget, ks)
            mine = [hashlib.sha256(t.cpu().numpy().astype(np.int64).tobytes()).hexdigest() for t in blocks[k]]
            assert mine == G[f"{tag}/block_digest"][ks], (budget, ks)
        sd = model3.state_dict()
        assert set(sd) == set(G[f"{tag}/digest"])
        for name, (shape, sha, s1, s2) in G[f"{tag}/digest"].items():
            assert tuple(sd[name].shape) == tuple(shape), (budget, name)
            assert _digest(sd[name])[0] == sha, (budget, name)


# ----------------------------------------------------------------------------------------- PLeaS train

def _train18_setup(P, G):
    m1, m2 = _pair("resnet18")
    spec = P.get_permutation_spec(m1, ((1, 3, 224, 224),))
    m1, m2 = m1.cuda(), m2.cuda()
    perm_mine, costs = P.activation_matching(spec, m1, m2, _loader(*G["am_loader"]), num_batches=2, output_costs=True)
    perm = {k: G["perm"][key_str(k)].to(torch.int64) for k in spec}
    assert all(torch.equal(perm[k], perm_mine[k]) for k in spec)
    return m1, m2, spec, perm, costs


def _logits_after_bn_reset(P, model3, G):
    P.reset_bn_stats(model3, _loader(*G["train_loader"]), num_batches=101, reset=True)
    xh = _loader(*G["heldout"])[0][0].cuda()
    with torch.no_grad():
        return model3(xh).float().cpu()


def _rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


@pytest.mark.parametrize("ridge,logit_tol", [(1e-4, 2e-3), (1e-6, 2e-2)])
def test_train_rn18_logits_closed_form_vs_fp64_lstsq(ridge, logit_tol):
    """ResNet-18 at 224x224, 41 batches of 16: the closed form (3xTF32 normal equations in fp64
    accumulators + fp64 Cholesky) against an fp64 ridge least squares built from the reference's own
    get_model_orig_activations pairs.  Logits of the fitted model after the drivers' BN reset on a
    held-out batch: rel-L2 <= 2e-3 at the default ridge 1e-4 (measured 1.4e-3; SURVEY 8c(6) proposed 1e-3, but
    the cuDNN-vs-oneDNN forward differences alone put the Adam replay below, which builds no normal
    equations at all, at 0.9e-3 on the same batches); with a ridge of 1e-6 the ill-conditioned layers (fc: 656 sample rows for 513 unknowns) amplify the fp32-level noise of the normal
    equations and the bar is 2e-2 (the two fp64 solutions themselves differ by 0.79 in the logits).
    Per-layer objective gain within 1e-3 of the fp64 one at either ridge."""
    P = _pkg()
    G = _load("train18_golden.pt")
    m1, m2, spec, perm, costs = _train18_setup(P, G)
    model3 = P.partial_merge(spec, m1, m2, perm, costs, 0.0)
    stats = {}
    P.train(_loader(*G["train_loader"]), m1, m2, model3, spec, perm, costs, 0.0, False, G["max_steps"], None,
            num_classes=1000, model_type="rn18", ridge=ridge, stats=stats)
    sd = model3.state_dict()
    for name, gs in G[f"layer_stats/{ridge:g}"].items():
        st = stats[name]
        gain_mine = (st["objective_fit"] - st["objective_init"]) / (st["rows"] * st["cout"])
        gain_gold = gs["loss_lstsq"] - gs["loss_init"]
        assert abs(gain_mine - gain_gold) <= 1e-3 * abs(gain_gold) + 1e-6, (name, gain_mine, gain_gold)
        assert st["ridge_rel"] == pytest.approx(ridge), name  # no pivot failure escalated the ridge
        W = sd[f"{name}.weight"].flatten(1).cpu()
        r, s = np.random.default_rng(7).integers(0, W.shape[0], 64), np.random.default_rng(8).integers(0, W.shape[1], 64)
        rms = gs["w_norm"] / np.sqrt(W.numel())
        err = float((W[torch.from_numpy(r), torch.from_numpy(s)] - gs["w_samples"]).abs().max())
        # sampled weight entries; a layer with few more sample rows than unknowns (fc: 656 rows, 513 unknowns)
        # is ill-conditioned, its weights are only pinned through the logits below
        assert err <= (2e-2 if st["rows"] >= 4 * st["K"] else 1e-1) * rms, (name, err, rms)
    logits = _logits_after_bn_reset(P, model3, G)
    gold = G[f"logits/lstsq/{ridge:g}"]
    err = _rel_l2(logits, gold)
    print(f"closed form vs fp64 lstsq (ridge {ridge:g}): logit rel-L2 {err:.2e} "
          f"(init vs lstsq {_rel_l2(G['logits/init'], gold):.2f})")
    assert err <= logit_tol


def test_train_rn18_logits_adam_replay_vs_reference():
    """solver="adam" replays the reference optimiser (pleas_merging.py:234-302, 357-397) for
    MAX_STEPS=40 on the same batches: logits after the BN reset within 5e-2 rel-L2 of the reference
    run's (cuDNN vs oneDNN forwards under Adam's sign-like steps)."""
    P = _pkg()
    G = _load("train18_golden.pt")
    m1, m2, spec, perm, costs = _train18_setup(P, G)
    model3 = P.partial_merge(spec, m1, m2, perm, costs, 0.0)
    P.train(_loader(*G["train_loader"]), m1, m2, model3, spec, perm, costs, 0.0, False, G["max_steps"], None,
            num_classes=1000, model_type="rn18", solver="adam")
    logits = _logits_after_bn_reset(P, model3, G)
    err = _rel_l2(logits, G["logits/adam"])
    print(f"adam replay vs reference: logit rel-L2 {err:.2e}")
    assert err <= 5e-2


# ----------------------------------------------------------------------------------------- config 4

def test_config4_rn101_domainnet_vs_oracle():
    """BASELINE config 4's model pair — ResNet-101 with the 345-class DomainNet head
    (experiments/shared_label_space/run_domainnet.py:182-186), 71 permutation groups, 344 taps — on one batch of
    4 x 224x224 (the oracle port's CPU forward bounds the size): cost matrices within the 1e-4 bar of the oracle and
    identical permutations (or an equal optimum within 1e-6 on the oracle's costs); the spec equals the reference's
    (tests/golden/spec_resnet101.json; the head changes no permutation group)."""
    import torchvision

    P = _pkg()

    def build(seed):
        torch.manual_seed(seed)
        m = torchvision.models.resnet101()
        m.fc = torch.nn.Linear(2048, 345)
        return m.eval()

    m1, m2 = build(0), build(1)
    spec = P.get_permutation_spec(m1, ((1, 3, 224, 224),))
    jspec = load_spec_json("resnet101")
    assert [(k.key, k.axis, pg.size) for k, pg in spec.items()] == [(g["key"][0], g["key"][1], g["size"]) for g in jspec]
    g = torch.Generator().manual_seed(123)
    loader = [(torch.randn(4, 3, 224, 224, generator=g), 0)]
    ocosts = O.matching_costs(jspec, m1, m2, loader, 1, "cdist", "sum")
    perm, costs = P.activation_matching(spec, m1.cuda(), m2.cuda(), loader, 1, output_costs=True)
    flips, worst = 0, 0.0
    for k in spec:
        oc = ocosts[(k.key, k.axis)]
        worst = max(worst, _relerr(costs[k].cpu().numpy(), oc))
        operm, _ = O.solve_lsa(oc, True)
        flips += _perm_or_objective(perm[k].numpy(), operm, oc, str(k))
    assert worst <= 1e-4
    print(f"config 4 (ResNet-101 / 345 classes): max cost rel-err {worst:.2e}; assignments differing from the oracle: "
          f"{flips} of {sum(pg.size for pg in spec.values())}")
