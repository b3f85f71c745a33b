"""Method-level parity: the drop-in API on the B200 against the golden outputs of the
unmodified reference (tests/golden/) and the CPU oracle."""
import copy

import numpy as np
import pytest
import torch

from conftest import key_str, load_spec_json
from oracle import ref_oracle as O
from oracle import tinynet

pytestmark = pytest.mark.gpu


def _pkg():
    import pleas_merging_b200 as P

    return P


def _tiny(P):
    m1, m2 = tinynet.make_pair(12, 10)
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    return m1.cuda(), m2.cuda(), spec


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def assert_perm_or_objective(perm, gold_perm, cost, name):
    """Identical permutation, else an equal optimum (rel 1e-6) on the reference's cost matrix."""
    perm, gold_perm = np.asarray(perm), np.asarray(gold_perm)
    if (perm == gold_perm).all():
        return
    c = np.asarray(cost, dtype=np.float64)
    idx = np.arange(len(perm))
    a, b = c[idx, perm].sum(), c[idx, gold_perm].sum()
    assert abs(a - b) <= 1e-6 * abs(b), f"{name}: objective {a} vs reference {b}"


@pytest.mark.parametrize("cross", ["cdist", "inner"])
@pytest.mark.parametrize("accumulate", ["reference", "sum"])
def test_activation_matching_tiny_vs_reference(tiny_golden, cross, accumulate):
    P = _pkg()
    m1, m2, spec = _tiny(P)
    loader = tinynet.make_loader(*tiny_golden["loader"])
    cf = P.cross_features_cdist if cross == "cdist" else P.cross_features_inner_product
    perm, costs = P.activation_matching(spec, m1, m2, loader, len(loader), cross_features=cf, output_costs=True,
                                        accumulate=accumulate)
    gp, gc = tiny_golden[f"am/{cross}/{accumulate}/perm"], tiny_golden[f"am/{cross}/{accumulate}/costs"]
    assert list(perm.keys()) == list(spec.keys())
    for k in spec:
        assert perm[k].dtype == torch.int64 and not perm[k].is_cuda and costs[k].is_cuda
        assert relerr(costs[k].cpu().numpy(), gc[key_str(k)].numpy()) <= 1e-4, k  # north-star matrix bar
        assert_perm_or_objective(perm[k].numpy(), gp[key_str(k)].numpy(), gc[key_str(k)].numpy(), k)
        assert (perm[k].numpy() == gp[key_str(k)].numpy()).all(), k  # no ties in this fixture


def test_plugin_operators_in_generic_path(tiny_golden):
    """The library's operators satisfy the reference's plug-in signatures: used through the
    generic (un-fused) path with a user wrapper they reproduce the fused result."""
    P = _pkg()
    import importlib

    AM = importlib.import_module("pleas_merging_b200.methods.activation_matching")

    m1, m2, spec = _tiny(P)
    loader = tinynet.make_loader(*tiny_golden["loader"])

    def my_cross(x, y, a):
        return P.cross_features_cdist(x, y, a)

    def my_solver(A, maximize=True):
        return P.b200_solve_lsa(A, maximize)

    perm, costs = P.activation_matching(spec, m1, m2, loader, len(loader), cross_features=my_cross,
                                        lsa_solver=my_solver, output_costs=True, accumulate="sum")
    for k in spec:
        assert relerr(costs[k].cpu().numpy(), tiny_golden["am/cdist/sum/costs"][key_str(k)].numpy()) <= 1e-4
        assert (perm[k].numpy() == tiny_golden["am/cdist/sum/perm"][key_str(k)].numpy()).all()
    # build_cross_module returns the reference's structure
    axes = [ax for pg in spec.values() for ax in pg.node]
    gm = AM.build_cross_module(m1, m2, axes, my_cross)
    with torch.inference_mode():
        (o1, o2), cross = gm(loader[-1][0].cuda())
    assert o1.shape == o2.shape == (4, 10) and len(cross) == 22
    gold = tiny_golden["am/cdist/taps_last"]
    for (name, axis), v in cross.items():
        assert relerr(v.cpu().numpy(), gold[f"{name}:{axis}"].numpy()) <= 1e-4


def test_weight_matching_tiny_vs_reference(tiny_golden):
    P = _pkg()
    m1, m2, spec = _tiny(P)
    sd2 = m2.state_dict()
    before = {k: v.clone() for k, v in sd2.items()}
    perm, costs = P.weight_matching(spec, m1.state_dict(), sd2, max_iter=100, seed=0, verbose=False,
                                    return_costs=True)
    for k in spec:
        assert (perm[k].numpy() == tiny_golden["wm/perm"][key_str(k)].numpy()).all(), k
        assert relerr(costs[k].cpu().numpy(), tiny_golden["wm/costs"][key_str(k)].numpy()) <= 1e-5, k
    assert all(torch.equal(sd2[k], before[k]) for k in before)  # inplace=False leaves B untouched


@pytest.mark.parametrize("name", ["r0", "r05", "r1", "mixed"])
def test_partial_merge_tiny_vs_reference(tiny_golden, name):
    P = _pkg()
    m1, m2, spec = _tiny(P)
    perm = {k: tiny_golden["am/cdist/sum/perm"][key_str(k)] for k in spec}
    costs = {k: tiny_golden["am/cdist/sum/costs"][key_str(k)].cuda() for k in spec}
    r = tiny_golden[f"pm/{name}/ratios"]
    ratios = {k: r[key_str(k)] for k in spec} if isinstance(r, dict) else r
    model3, blocks = P.partial_merge(spec, m1, m2, perm, costs, ratios, return_blocks=True)
    for k in spec:
        for mine, gold in zip(blocks[k], tiny_golden[f"pm/{name}/blocks"][key_str(k)]):
            assert mine.dtype == torch.int64 and torch.equal(mine.cpu(), gold)
    gold_state = tiny_golden[f"pm/{name}/state"]
    sd3 = model3.state_dict()
    assert set(sd3.keys()) == set(gold_state.keys())
    for k, v in gold_state.items():
        assert torch.equal(sd3[k].cpu(), v), k  # gathers and (a+b)/2: bit exact
    assert not model3.training
    assert all(not dict(model3.named_parameters())[k].requires_grad for k in gold_state if k in dict(model3.named_parameters()) and k != 'fc.bias')
    with torch.no_grad():  # the merged module is runnable
        assert model3(torch.randn(2, 3, 16, 16).cuda()).shape == (2, 10)


def _merged_init(P, tiny_golden, name, m1, m2, spec):
    perm = {k: tiny_golden["am/cdist/sum/perm"][key_str(k)] for k in spec}
    costs = {k: tiny_golden["am/cdist/sum/costs"][key_str(k)].cuda() for k in spec}
    ratios = tiny_golden[f"pm/{name}/ratios"]
    return perm, costs, ratios, P.partial_merge(spec, m1, m2, perm, costs, ratios)


@pytest.mark.parametrize("name", ["r0", "r05"])
def test_train_closed_form_vs_reference(tiny_golden, name):
    """Per-layer objective of the closed form: matches the fp64 optimum computed from the
    reference's own (X-bar, Y-bar) pairs and is never worse than the reference's Adam result."""
    P = _pkg()
    m1, m2, spec = _tiny(P)
    perm, costs, ratios, model3 = _merged_init(P, tiny_golden, name, m1, m2, spec)
    loader = tinynet.make_loader(*tiny_golden["train/loader"])
    steps = tiny_golden["train/max_steps"]
    stats = {}
    # ridge 1e-6: the golden optimum is the ridge-free minimum-norm update (pinv), the default 1e-4 trades
    # a few percent of the calibration objective of the tiny fc layer for conditioning
    out = P.train(loader, m1, m2, model3, spec, perm, costs, ratios, False, steps, None, num_classes=10,
                  model_type="rn18", stats=stats, ridge=1e-6)
    assert out is model3
    # evaluate the fitted weights with the CPU oracle's fp64 normal equations
    jspec = load_spec_json("tiny")
    c1, c2 = tinynet.make_pair(12, 10)
    ob = O.get_blocks(jspec, {g["key"]: perm[P.Axis(*g["key"])].numpy() for g in jspec},
                      {g["key"]: costs[P.Axis(*g["key"])].cpu().numpy() for g in jspec},
                      {g["key"]: ratios for g in jspec} if not isinstance(ratios, dict) else ratios)
    acc = O.pleas_normal_equations(jspec, c1, c2, ob, loader, steps, num_classes=10)
    sd3 = {k: v.detach().cpu().numpy() for k, v in model3.state_dict().items()}
    gold = tiny_golden[f"train/{name}/layer_stats"]
    for n, d in acc.items():
        mine = O.layer_loss(O.flat_weight(sd3, n, f"{n}.bias" in sd3), d)
        assert mine <= gold[n]["loss_adam"] * (1 + 1e-4) + 1e-9, (n, mine, gold[n])
        assert mine <= gold[n]["loss_lstsq"] * (1 + 2e-2) + 1e-7, (n, mine, gold[n])
        assert stats[n]["objective_fit"] <= stats[n]["objective_init"] + 1e-9
    assert set(stats["_timing"]) == {"accumulate_s", "solve_s"}


def _oracle_layer_losses(P, tiny_golden, perm, costs, ratios, model3):
    jspec = load_spec_json("tiny")
    c1, c2 = tinynet.make_pair(12, 10)
    loader = tinynet.make_loader(*tiny_golden["train/loader"])
    ob = O.get_blocks(jspec, {g["key"]: perm[P.Axis(*g["key"])].numpy() for g in jspec},
                      {g["key"]: costs[P.Axis(*g["key"])].cpu().numpy() for g in jspec}, ratios)
    acc = O.pleas_normal_equations(jspec, c1, c2, ob, loader, tiny_golden["train/max_steps"], num_classes=10)
    sd3 = {k: v.detach().cpu().numpy() for k, v in model3.state_dict().items()}
    return {n: O.layer_loss(O.flat_weight(sd3, n, f"{n}.bias" in sd3), d) for n, d in acc.items()}


def test_train_adam_replays_reference(tiny_golden):
    """solver="adam" follows the reference trajectory: same per-layer losses, and the same
    weights wherever the gradient is not rounding noise (conv1 is solved exactly by the init, so
    Adam's sign-like steps there are noise-driven on any platform)."""
    P = _pkg()
    m1, m2, spec = _tiny(P)
    perm, costs, ratios, model3 = _merged_init(P, tiny_golden, "r05", m1, m2, spec)
    loader = tinynet.make_loader(*tiny_golden["train/loader"])
    P.train(loader, m1, m2, model3, spec, perm, costs, ratios, False, tiny_golden["train/max_steps"], None,
            num_classes=10, model_type="rn18", solver="adam")
    gold_state = tiny_golden["train/r05/adam_state"]
    gold = tiny_golden["train/r05/layer_stats"]
    for n, mine in _oracle_layer_losses(P, tiny_golden, perm, costs, ratios, model3).items():
        assert mine == pytest.approx(gold[n]["loss_adam"], rel=2e-2, abs=1e-6), n
    for k, v in model3.state_dict().items():
        if not k.startswith("conv1."):
            assert torch.allclose(v.cpu(), gold_state[k], rtol=1e-2, atol=2e-4), k


def test_activation_matching_rn18_vs_reference(rn18_golden):
    import torchvision

    P = _pkg()
    torch.manual_seed(0)
    m1 = torchvision.models.resnet18().eval()
    torch.manual_seed(1)
    m2 = torchvision.models.resnet18().eval()
    spec = P.get_permutation_spec(m1, ((1, 3, 64, 64),))
    nb, b, hw, seed = rn18_golden["loader"]
    g = torch.Generator().manual_seed(seed)
    loader = [(torch.randn(b, 3, hw, hw, generator=g), 0) for _ in range(nb)]
    # oracle costs on the same inputs (CPU forward) to judge near-ties
    ocosts = O.matching_costs(load_spec_json("resnet18"), m1, m2, loader, nb, "cdist", "sum")
    perm, costs = P.activation_matching(spec, m1.cuda(), m2.cuda(), loader, nb, output_costs=True, accumulate="sum")
    for k in spec:
        ks = key_str(k)
        assert relerr(costs[k].cpu().numpy(), ocosts[(k.key, k.axis)]) <= 1e-4, k
        assert_perm_or_objective(perm[k].numpy(), rn18_golden["am/cdist/sum/perm"][ks].numpy().astype(np.int64),
                                 ocosts[(k.key, k.axis)], ks)


def test_planted_permutation_is_recovered():
    """Merging a model with a permuted copy of itself: both matchers recover the planted
    permutation and the ratio-0 merge reproduces the original function (SURVEY.md §4 (iii))."""
    P = _pkg()
    m1, _ = tinynet.make_pair(12, 10)
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    planted = P.make_random_perm(spec, generator=torch.Generator().manual_seed(9))
    m2 = copy.deepcopy(m1)
    P.apply_perm(planted, spec, m2, inplace=True)
    m1, m2 = m1.cuda(), m2.cuda()
    x = torch.randn(4, 3, 16, 16, generator=torch.Generator().manual_seed(10))
    with torch.no_grad():
        assert torch.allclose(m1(x.cuda()), m2(x.cuda()), rtol=1e-4, atol=1e-5)
    loader = [(x, 0)]
    inv = P.invert_perm(planted)
    perm_am, costs = P.activation_matching(spec, m1, m2, loader, 1, output_costs=True)
    perm_wm = P.weight_matching(spec, m1.state_dict(), m2.state_dict(), verbose=False)
    for k in spec:
        assert torch.equal(perm_am[k], inv[k]), k
        assert torch.equal(perm_wm[k], inv[k]), k
    merged = P.partial_merge(spec, m1, m2, perm_am, costs, 0.0)
    with torch.no_grad():
        assert torch.allclose(merged(x.cuda()), m1(x.cuda()), rtol=1e-4, atol=1e-5)


def test_two_gpu_sharded_paths_match_single_gpu():
    """Batch-sharded activation matching and PLeaS (NCCL all-reduce of the accumulators) give the
    single-GPU result.  Needs >= 2 GPUs; the host-side logic is covered on CPU with gloo."""
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    here = os.path.dirname(os.path.abspath(__file__))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(here, "dist_check.py")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "dist_check ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_activation_matching_rn50_full_width_vs_oracle():
    """Full-width ResNet-50 (groups up to 2048 units, 174 taps) on one 224x224 batch: cost
    matrices within the 1e-4 bar of the CPU oracle and identical permutations (or an equal
    optimum within 1e-6 on the oracle's costs)."""
    import torchvision

    P = _pkg()
    torch.manual_seed(0)
    m1 = torchvision.models.resnet50().eval()
    torch.manual_seed(1)
    m2 = torchvision.models.resnet50().eval()
    spec = P.get_permutation_spec(m1, ((1, 3, 224, 224),))
    g = torch.Generator().manual_seed(123)
    loader = [(torch.randn(4, 3, 224, 224, generator=g), 0)]
    ocosts = O.matching_costs(load_spec_json("resnet50"), m1, m2, loader, 1, "cdist", "sum")
    perm, costs = P.activation_matching(spec, m1.cuda(), m2.cuda(), loader, 1, output_costs=True)
    flips = 0
    for k in spec:
        oc = ocosts[(k.key, k.axis)]
        assert relerr(costs[k].cpu().numpy(), oc) <= 1e-4, k
        operm, _ = O.solve_lsa(oc, True)
        assert_perm_or_objective(perm[k].numpy(), operm, oc, str(k))
        flips += int((perm[k].numpy() != operm).sum())
    print("rn50 assignments differing from the oracle:", flips)


def _jspec(P, spec):
    return [{"key": (k.key, k.axis), "size": pg.size, "state": sorted((a.key, a.axis) for a in pg.state),
             "node": sorted((a.key, a.axis) for a in pg.node)} for k, pg in spec.items()]


@pytest.mark.parametrize("accumulate", ["reference", "sum"])
def test_ragged_batches_and_short_loader(accumulate):
    """Batches of different sizes (each shape gets its own CUDA graph) and num_batches larger than
    the loader (the reference's zip stops at the shorter one)."""
    P = _pkg()
    m1, m2 = tinynet.make_pair(12, 10)
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    g = torch.Generator().manual_seed(77)
    loader = [(torch.randn(b, 3, 16, 16, generator=g), 0) for b in (4, 4, 4, 3, 4, 3, 1)]
    operm, ocosts = O.activation_matching(_jspec(P, spec), m1, m2, loader, 50, "cdist", accumulate)
    perm, costs = P.activation_matching(spec, m1.cuda(), m2.cuda(), loader, 50, output_costs=True,
                                        accumulate=accumulate)
    for k in spec:
        assert relerr(costs[k].cpu().numpy(), ocosts[(k.key, k.axis)]) <= 1e-4, k
        assert_perm_or_objective(perm[k].numpy(), operm[(k.key, k.axis)], ocosts[(k.key, k.axis)], str(k))


def test_models_in_train_mode_use_batch_statistics():
    """The reference's drivers never call .eval() before activation matching (SURVEY 3.2): BN then
    normalises with batch statistics and updates its running stats.  The user's modules are run
    unchanged, eagerly and under CUDA-graph replay."""
    P = _pkg()
    a1, a2 = tinynet.make_pair(12, 10)
    b1, b2 = copy.deepcopy(a1), copy.deepcopy(a2)
    for m in (a1, a2, b1, b2):
        m.train()
    spec = P.get_permutation_spec(copy.deepcopy(a1).eval(), ((1, 3, 16, 16),))
    loader = tinynet.make_loader(4, 6, 16, seed=8)
    operm, ocosts = O.activation_matching(_jspec(P, spec), a1, a2, loader, 4, "cdist", "sum")
    g1, g2 = b1.cuda(), b2.cuda()
    perm, costs = P.activation_matching(spec, g1, g2, loader, 4, output_costs=True, accumulate="sum")
    for k in spec:
        assert relerr(costs[k].cpu().numpy(), ocosts[(k.key, k.axis)]) <= 1e-4, k
        assert_perm_or_objective(perm[k].numpy(), operm[(k.key, k.axis)], ocosts[(k.key, k.axis)], str(k))
    # running statistics advanced exactly like on the CPU (4 batches each)
    for (n, p), (_, q) in zip(a1.named_buffers(), g1.named_buffers()):
        assert torch.allclose(p, q.cpu(), rtol=1e-4, atol=1e-5), n


def test_train_with_ragged_last_batch_and_graphs_off():
    """Closed form with a ragged last batch equals the eager (no CUDA graph) run."""
    P = _pkg()
    m1, m2, spec = _tiny(P)
    g = torch.Generator().manual_seed(5)
    loader = [(torch.randn(b, 3, 16, 16, generator=g), 0) for b in (4, 4, 4, 4, 2)]
    perm, costs = P.activation_matching(spec, m1, m2, loader, 5, output_costs=True, accumulate="sum")
    outs = []
    for graphs in (True, False):
        m3 = P.partial_merge(spec, m1, m2, perm, costs, 0.3)
        P.train(loader, m1, m2, m3, spec, perm, costs, 0.3, False, 10, None, num_classes=10, model_type="rn18",
                use_cuda_graph=graphs)
        outs.append({k: v.clone() for k, v in m3.state_dict().items()})
    for k in outs[0]:
        assert torch.allclose(outs[0][k], outs[1][k], rtol=1e-5, atol=1e-7), k


@pytest.mark.parametrize("reset", [True, False])
def test_reset_bn_stats_matches_driver_loop(reset):
    """BN re-estimation equals the reference drivers' loop (run_domainnet.py:327-341) run on CPU."""
    P = _pkg()
    m, _ = tinynet.make_pair(12, 10)
    ref = copy.deepcopy(m)
    loader = tinynet.make_loader(6, 4, 16, seed=3)
    ref.train()
    if reset:
        for mod in ref.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.reset_running_stats()
    with torch.no_grad():
        for idx, (x, _) in enumerate(loader):
            ref(x)
            if idx + 1 >= 5:
                break
    out = P.reset_bn_stats(m.cuda(), loader, num_batches=5, reset=reset)
    assert out is m and not m.training
    for (n, a), (_, b) in zip(ref.named_buffers(), m.named_buffers()):
        assert torch.allclose(a, b.cpu().to(a.dtype), rtol=1e-4, atol=1e-6), n


def test_readme_basic_usage_flow_runs():
    """The reference README flow (spec -> AM -> partial_merge -> PLeaS -> BN reset) end to end."""
    import importlib.util
    import os

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "basic_usage.py")
    spec = importlib.util.spec_from_file_location("basic_usage", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    model, stats = mod.main("resnet18", num_batches=3, batch=4, hw=64, max_steps=3, verbose=False)
    layers = [k for k in stats if not k.startswith("_")]
    assert len(layers) == 21 and all(stats[k]["objective_fit"] <= stats[k]["objective_init"] + 1e-6 for k in layers)
    with torch.no_grad():
        assert bool(torch.isfinite(model(torch.randn(2, 3, 64, 64).cuda())).all())


@pytest.mark.parametrize("merging,ratio", [("perm_separatels", 0.5), ("perm_mixedls", 0.5), ("reg_mean", 0.0),
                                           ("perm_gradmask", 0.5)])
def test_closed_form_alternative_targets(merging, ratio):
    """The closed form on the reference's alternative least-squares targets (pleas_merging.py:125-147):
    per layer, its objective equals the fp64 optimum of the explicitly stacked (X-bar, Y-bar) problem
    built with the torch restatement of get_model_orig_activations, masked entries held at the init."""
    import importlib
    import torch.nn.functional as F

    P = _pkg()
    PM = importlib.import_module("pleas_merging_b200.methods.pleas_merging")
    m1, m2, spec = _tiny(P)
    loader = tinynet.make_loader(6, 4, 16, seed=21)
    perm, costs = P.activation_matching(spec, m1, m2, loader, 6, output_costs=True, accumulate="sum")
    model3 = P.partial_merge(spec, m1, m2, perm, costs, ratio)
    init = {k: v.detach().clone() for k, v in model3.state_dict().items()}
    P.train(loader, m1, m2, model3, spec, perm, costs, ratio, False, 5, None, num_classes=10, model_type="rn18",
            merging=merging)
    fitted = model3.state_dict()
    # explicit fp64 problem
    blocks = P.get_blocks(spec, perm, costs, ratio)
    pb = dict(blocks)
    for axis, pg in spec.items():
        for ax in pg.state:
            pb[ax] = pb[axis]
    a1, a2 = {}, {}
    hooks = PM.capture_inputs(m1, a1) + PM.capture_inputs(m2, a2)
    Us, Ts = {}, {}
    with torch.no_grad():
        for x, _ in loader:
            m1(x.cuda())
            m2(x.cuda())
            for name, layer in m1.named_modules():
                if not isinstance(layer, (torch.nn.Conv2d, torch.nn.Linear)):
                    continue
                bi, bo = PM._layer_blocks(pb, name, a1[name][0].shape[1], 10, False, "rn18")
                X, Y = PM.get_model_orig_activations(a1[name], a2[name], bi, bo, merging)
                X, Y = X.double(), Y.double()
                if isinstance(layer, torch.nn.Conv2d):
                    U = F.unfold(X, layer.kernel_size, layer.dilation, layer.padding, layer.stride)
                    U = U.transpose(1, 2).reshape(-1, U.shape[1])
                    T = Y.flatten(2).transpose(1, 2).reshape(-1, Y.shape[1])
                else:
                    U, T = X, Y
                if layer.bias is not None:
                    U = torch.cat([U, torch.ones(U.shape[0], 1, dtype=U.dtype, device=U.device)], 1)
                Us.setdefault(name, []).append(U)
                Ts.setdefault(name, []).append(T)
    for h in hooks:
        h.remove()
    for name in Us:
        U, T = torch.cat(Us[name]), torch.cat(Ts[name])

        def flat(sd):
            W = sd[f"{name}.weight"].double().flatten(1)
            return torch.cat([W, sd[f"{name}.bias"].double()[:, None]], 1) if f"{name}.bias" in sd else W

        W0, Wf = flat(init), flat(fitted)
        loss = lambda W: float(((U @ W.T - T) ** 2).sum())
        # fp64 optimum: minimum-norm update from W0 (unmasked layers only keeps this check simple)
        dW = torch.linalg.lstsq(U.cpu(), (T - U @ W0.T).cpu(), driver="gelsd").solution.T.to(U.device)  # rank-deficient U
        best = loss(W0 + dW)
        scale = float((T ** 2).sum()) + 1e-12
        assert loss(Wf) <= loss(W0) + 1e-9 * scale, name
        if ratio == 0.0 or merging != "perm_gradmask":
            # no gradient mask constraints bite at ratio 0; for ratio 0.5 masked rows make `best` a lower bound
            assert loss(Wf) >= best - 1e-6 * scale, name
        if ratio == 0.0:
            assert loss(Wf) <= best + 2e-3 * scale, name


def test_full_size_properties_rn50():
    """BASELINE config-2 sizes (ResNet-50, batches of 32x3x224x224), where the CPU oracle is too
    slow: (1) a model matched against a permuted copy of itself recovers the planted permutation in
    every one of the 37 groups; (2) accumulate="sum" is linear over batches; (3) accumulate=
    "reference" equals the last batch alone."""
    import torchvision

    P = _pkg()
    torch.manual_seed(0)
    m1 = torchvision.models.resnet50().eval()
    spec = P.get_permutation_spec(m1, ((1, 3, 224, 224),))
    planted = P.make_random_perm(spec, generator=torch.Generator().manual_seed(3))
    m2 = copy.deepcopy(m1)
    P.apply_perm(planted, spec, m2, inplace=True)
    m1, m2 = m1.cuda(), m2.cuda()
    g = torch.Generator().manual_seed(4)
    loader = [(torch.randn(32, 3, 224, 224, generator=g), 0) for _ in range(3)]
    perm, c_all = P.activation_matching(spec, m1, m2, loader, 3, output_costs=True, accumulate="sum")
    inv = P.invert_perm(planted)
    for k in spec:
        assert torch.equal(perm[k], inv[k]), k
    parts = [P.activation_matching(spec, m1, m2, [b], 1, output_costs=True, accumulate="sum")[1] for b in loader]
    _, c_ref = P.activation_matching(spec, m1, m2, loader, 3, output_costs=True)  # reference semantics
    for k in spec:
        total = parts[0][k] + parts[1][k] + parts[2][k]
        scale = float(total.abs().max())
        assert float((c_all[k] - total).abs().max()) <= 2e-6 * scale, k
        assert float((c_ref[k] - parts[2][k]).abs().max()) <= 2e-6 * float(parts[2][k].abs().max()), k


@pytest.mark.parametrize("name", ["r0", "r05", "r1", "mixed"])
def test_get_fc_perm_equals_reference(tiny_golden, eval_golden, name):
    """SURVEY 8f n3: the classifier group's blocks (pleas_merging.py:408-433) equal the reference's."""
    P = _pkg()
    from pleas_merging_b200.methods.evaluation import get_fc_perm, permute_final_features

    _, _, spec = _tiny(P)
    perm = {k: tiny_golden["am/cdist/sum/perm"][key_str(k)] for k in spec}
    costs = {k: tiny_golden["am/cdist/sum/costs"][key_str(k)].cuda() for k in spec}
    r = eval_golden[f"{name}/ratios"]
    ratios = {k: r[key_str(k)] for k in spec} if isinstance(r, dict) else r
    fc_perm = get_fc_perm(perm, spec, costs, ratios)
    for mine, gold in zip(fc_perm, eval_golden[f"{name}/fc_perm"]):
        assert torch.equal(mine.cpu(), gold)
    feats = eval_golden[f"{name}/features"].cuda()
    for idx in (0, 1):
        assert torch.equal(permute_final_features(feats, fc_perm, idx).cpu(), eval_golden[f"{name}/out{idx}"])


@pytest.mark.parametrize("ratio", [0.0, 0.5])
def test_eval_perm_model_recovers_source_predictions(ratio):
    """Merging a network with a hidden-unit-permuted copy of itself is lossless, so the merged
    backbone (fc removed) + either source classifier must score exactly what that source model
    scores on its own labels — checks get_fc_perm / permute_final_features / eval_perm_model /
    eval_whole_model end to end (pleas_merging.py:408-496, 574-585)."""
    P = _pkg()
    from pleas_merging_b200.methods import evaluation as E

    m1, _ = tinynet.make_pair(12, 10)
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    planted = P.make_random_perm(spec, torch.Generator().manual_seed(3))
    m2 = copy.deepcopy(m1)
    m2.load_state_dict(P.apply_perm(planted, spec, m1.state_dict()))
    m1, m2 = m1.cuda(), m2.cuda()
    loader = tinynet.make_loader(3, 8, 16)
    perm, costs = P.activation_matching(spec, m1, m2, loader, 3, output_costs=True, accumulate="sum")
    model3 = P.partial_merge(spec, m1, m2, perm, costs, ratio).cuda()
    fc_perm = E.get_fc_perm(perm, spec, costs, ratio)
    # labels = model 1's own predictions -> accuracy of model 1 is 1.0 by construction
    with torch.no_grad():
        data = [(x, m1(x.cuda()).argmax(1).cpu()) for x, _ in tinynet.make_loader(4, 8, 16, seed=9)]
    assert float(E.eval_whole_model(m1, data, 10)) == 1.0
    backbone = copy.deepcopy(model3)
    backbone.fc = torch.nn.Identity()
    for idx, src in enumerate((m1, m2)):
        acc = E.eval_perm_model(backbone, src.fc, data, 10, fc_perm, idx)
        assert float(acc) == 1.0, (ratio, idx, float(acc))


@pytest.mark.parametrize("name", ["r05", "mixed"])
def test_weight_matching_partial_gpu_equals_reference(name):
    """weight_matching_partial with the product plug-ins (GPU LAP, tcgen05 Gram) on CUDA state dicts
    reproduces the reference's permutation and expanded state dicts (tests/golden/wmp_golden.pt)."""
    import os

    from conftest import GOLDEN
    from pleas_merging_b200.methods import weight_matching_partial

    P = _pkg()
    G = torch.load(os.path.join(GOLDEN, "wmp_golden.pt"), weights_only=False)
    m1, m2 = tinynet.make_pair(12, 10)
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    ratios = {k: G[f"{name}/ratios"][key_str(k)] for k in spec}
    sa = {k: v.clone().cuda() for k, v in m1.state_dict().items()}
    sb = {k: v.clone().cuda() for k, v in m2.state_dict().items()}
    perm = weight_matching_partial(spec, sa, sb, ratios, max_iter=20, inplace=True, verbose=False, seed=0)
    for k in spec:
        assert torch.equal(perm[k].cpu(), G[f"{name}/perm"][key_str(k)]), k
    for tag, mine in (("state_a", sa), ("state_b", sb)):
        for k, v in G[f"{name}/{tag}"].items():
            assert torch.equal(mine[k].cpu(), v), (tag, k)  # gathers and zero blocks only: bit exact


@pytest.mark.parametrize("accumulate", ["reference", "sum"])
def test_activation_matching_correlation_statistic(accumulate):
    """cross_features_correlation through the fused accumulation loop and through the generic plug-in path:
    cost matrices equal the oracle's float64 numpy.corrcoef restatement, permutations identical or an equal
    optimum on the oracle's costs.  The kernel-level bar (identical activations) is 2e-5, tests/test_kernels_gpu.py;
    end to end the statistic itself amplifies the ~1e-7 cuDNN-vs-oneDNN activation differences on nearly
    constant units (variance = difference of two large moments), hence 1e-3 absolute on sums of up to 4 taps."""
    P = _pkg()
    m1, m2 = tinynet.make_pair(12, 10)
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    loader = tinynet.make_loader(3, 8, 16, seed=31)
    operm, ocosts = O.activation_matching(_jspec(P, spec), m1, m2, loader, 3, "corr", accumulate)
    g1, g2 = m1.cuda(), m2.cuda()
    perm, costs = P.activation_matching(spec, g1, g2, loader, 3, cross_features=P.cross_features_correlation,
                                        output_costs=True, accumulate=accumulate)

    def wrapped(x, y, a):  # an unknown callable takes the generic (un-fused) path
        return P.cross_features_correlation(x, y, a)

    perm2, costs2 = P.activation_matching(spec, g1, g2, loader, 3, cross_features=wrapped, output_costs=True,
                                          accumulate=accumulate)
    for k in spec:
        oc = ocosts[(k.key, k.axis)]
        assert np.abs(costs[k].cpu().numpy() - oc).max() <= 1e-3, k
        assert np.abs(costs2[k].cpu().numpy() - oc).max() <= 1e-3, k
        # fused loop == generic plug-in path, up to the BatchNorm layers: the fused loop folds them into the convolution
        # launch and derives their taps from the tap in front (sign(s_a s_b) corr, exact), the plug-in runs the modules
        # and contracts the shifted fp32 outputs (variance by cancellation); both are within 1e-3 of the fp64 oracle
        assert (costs[k] - costs2[k]).abs().max() <= 1e-3, k
        assert_perm_or_objective(perm[k].numpy(), operm[(k.key, k.axis)], oc, str(k))
        assert_perm_or_objective(perm2[k].numpy(), operm[(k.key, k.axis)], oc, str(k))


def test_models_on_a_non_current_device():
    """Tensors on cuda:1 while cuda:0 is the current device (plain ``model.to('cuda:1')``, which the reference
    handles): every C-ABI call must be issued with the tensors' device current and on its stream.  Needs 2 GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    P = _pkg()
    m1, m2 = tinynet.make_pair(12, 10)
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    loader = tinynet.make_loader(3, 4, 16)
    assert torch.cuda.current_device() == 0
    ref_perm, ref_costs = P.activation_matching(spec, copy.deepcopy(m1).cuda(0), copy.deepcopy(m2).cuda(0), loader, 3,
                                                output_costs=True, accumulate="sum")
    a, b = m1.to("cuda:1"), m2.to("cuda:1")
    perm, costs = P.activation_matching(spec, a, b, loader, 3, output_costs=True, accumulate="sum")
    assert torch.cuda.current_device() == 0
    for k in spec:
        assert costs[k].device == torch.device("cuda", 1)
        assert torch.equal(perm[k], ref_perm[k]), k
        assert float((costs[k].cpu() - ref_costs[k].cpu()).abs().max()) <= 2e-6 * float(ref_costs[k].abs().max()), k
    merged = P.partial_merge(spec, a, b, perm, costs, 0.5)
    P.train(loader, a, b, merged, spec, perm, costs, 0.5, False, 2, None, num_classes=10, model_type="rn18")
    wperm = P.weight_matching(spec, a.state_dict(), b.state_dict(), verbose=False)
    wref = P.weight_matching(spec, m1.to("cuda:0").state_dict(), m2.to("cuda:0").state_dict(), verbose=False)
    assert all(torch.equal(wperm[k], wref[k]) for k in spec)


@pytest.mark.parametrize("mode", ["cdist", "inner", "corr"])
def test_batchnorm_taps_derived_from_the_tap_in_front_equal_contracted_taps(mode, monkeypatch):
    """An eval-mode BatchNorm tap is not contracted: its statistic is formed in the grouped epilogue from the Gram,
    row sums and sums of squares of the tap in front of it (PlbFinalizeTap.n_affine).  Same cost matrices as with
    every tap contracted (PLB_BN_AFFINE=0), negative BatchNorm scales included; fewer Gram launches."""
    import importlib

    from pleas_merging_b200 import _native

    AM = importlib.import_module("pleas_merging_b200.methods.activation_matching")
    P = _pkg()
    m1, m2 = tinynet.make_pair(12, 10)
    with torch.no_grad():
        m1.layer1[0].bn2.weight[::3] *= -1.0  # negative scales: the correlation flips sign per unit pair
        m2.layer2[0].bn1.weight[1::4] *= -1.0
    g1, g2 = m1.cuda(), m2.cuda()
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    loader = tinynet.make_loader(3, 8, 16, seed=7)
    fn = {"cdist": P.cross_features_cdist, "inner": P.cross_features_inner_product,
          "corr": P.cross_features_correlation}[mode]
    out = {}
    for flag in (True, False):
        monkeypatch.setattr(AM, "BN_AFFINE", flag)
        AM.clear_caches()
        _native.LAUNCH_COUNTS.clear()
        perm, costs = P.activation_matching(spec, g1, g2, loader, 3, cross_features=fn, output_costs=True,
                                            accumulate="sum", use_cuda_graph=False)
        out[flag] = (perm, costs, _native.LAUNCH_COUNTS["plb_gram_tma"] + _native.LAUNCH_COUNTS["plb_pack_split_pair"]
                     + _native.LAUNCH_COUNTS["plb_pack_split_pair_sums"])
    AM.clear_caches()
    assert out[True][2] < out[False][2]  # the BatchNorm taps launched nothing
    for k in spec:
        a, b = out[True][1][k], out[False][1][k]
        scale = float(b.abs().max())
        # correlation: the contracted BatchNorm tap forms variances of SHIFTED fp32 outputs by cancellation, the
        # derived one is sign(s_a s_b) corr of the tap in front — the difference is the contracted path's error
        assert float((a - b).abs().max()) <= (2e-3 if mode == "corr" else 1e-5 * scale), (k, mode)
        assert_perm_or_objective(out[True][0][k].numpy(), out[False][0][k].numpy(), b.cpu().numpy(), str(k))


def test_bench_dumps_the_timed_batches_costs(tmp_path):
    """`bench.py --dump-outputs DIR` on the B200 arm writes the cost matrices of the `--steps` timed batches alone —
    not the launch-count probe or the warm-up batches the benchmark's calibration runner sees first — i.e. what
    activation_matching(accumulate="sum") returns for those batches, recomputed here from the benchmark's seeded
    inputs (device generator 123, min(steps + warmup, 16) distinct batches, step i runs batch (warmup + i) mod that)."""
    import json
    import os
    import subprocess
    import sys

    import bench

    steps, warm = 3, 2
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--model", "resnet18", "--steps", str(steps),
                          "--warmup", str(warm), "--no-merge", "--no-cpu-baseline", "--no-extra-rooflines",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-3000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
    P = _pkg()
    m1, m2 = bench.make_models("resnet18", torch.device("cuda"))
    spec = P.get_permutation_spec(m1, ((1, 3, 224, 224),))
    gen = torch.Generator(device="cuda").manual_seed(123)
    dev = [torch.randn(32, 3, 224, 224, generator=gen, device="cuda") for _ in range(min(steps + warm, 16))]
    loader = [(dev[(warm + i) % len(dev)].cpu(), 0) for i in range(steps)]
    _, costs = P.activation_matching(spec, m1, m2, loader, steps, output_costs=True, accumulate="sum")
    assert sorted(f.name for f in tmp_path.iterdir()) == sorted(f"cost_{k.key}_{k.axis}.npy" for k in spec)
    for k in spec:
        got = np.load(tmp_path / f"cost_{k.key}_{k.axis}.npy")
        want = costs[k].cpu().numpy().astype(np.float64)
        assert got.dtype == np.float32 and got.shape == want.shape, k
        assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max(), k
