"""Golden outputs of the UNMODIFIED reference at the BASELINE.json config sizes (build container only).

TEST INFRASTRUCTURE ONLY.  Run as

    PYTHONHASHSEED=0 python -m oracle.make_golden_configs [cfg1] [cfg2] [cfg3] [train18]

(complements oracle/make_golden.py, whose fixtures are toy-sized).  Each section runs the
reference's public functions, imported from /root/reference through oracle/import_reference.py,
on seeded synthetic inputs at the sizes BASELINE.json names, and stores what a GPU-side test
needs to pin parity without the reference tree:

  cfg1_rn18_golden.pt   config 1: ResNet-18 pair, activation_matching on 10 batches of 32x3x224x224
                        (pleas/methods/activation_matching.py:139-177, verbatim last-batch semantics
                        and the accumulate-fixed sum), permutations, objectives and cost
                        fingerprints (the 4.2 MB of matrices are not stored: the tests recompute
                        them with the oracle port) + partial_merge ratio 0.0 state-dict digests
                        (pleas/methods/partial_matching.py:188-202)
  cfg2_rn50_golden.pt   config 2 (verbatim mode = the last batch alone): ResNet-50 pair, one batch
                        of 32x3x224x224 -> 37 permutations, objectives and cost fingerprints
                        (row / column sums, diagonal, sampled entries; the 32 MB of matrices are
                        not stored)
  cfg3_rn50_golden.pt   config 3: ResNet-50 weight_matching(seed=0) (pleas/methods/
                        weight_matching.py:22-95): permutations, LAP-call count, cost fingerprints;
                        partial_merge at budgets 1.2 / 1.55 / 1.8 / 2.0 with the drivers' zip rule
                        (experiments/different_label_space/run_torchvision.py:32-54): block sizes and
                        per-tensor digests
  train18_golden.pt     ResNet-18 at 224x224: reference Adam ``train`` (pleas/methods/
                        pleas_merging.py:305-405) for MAX_STEPS steps, the fp64 ridge least-squares
                        optimum built from the reference's own get_model_orig_activations pairs, and
                        the LOGITS of both after the drivers' BN reset
                        (experiments/shared_label_space/run_domainnet.py:327-341) on a held-out batch
"""
import hashlib
import os
import sys
import time

import numpy as np
import torch

from oracle.import_reference import accumulate_fixed_costs, load_reference

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
N_SAMPLES = 256


def axis_key(a):
    return f"{a.key}:{a.axis}"


def make_pair(arch, fc_out=None):
    import torchvision

    torch.manual_seed(0)
    m1 = getattr(torchvision.models, arch)().eval()
    torch.manual_seed(1)
    m2 = getattr(torchvision.models, arch)().eval()
    return m1, m2


def make_loader(nb, b, hw, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(b, 3, hw, hw, generator=g), 0) for _ in range(nb)]


def sample_index(n):
    """The sampled entries of an n x n cost matrix (seeded by n; the tests recompute them)."""
    rng = np.random.default_rng(1000 + n)
    return rng.integers(0, n, N_SAMPLES), rng.integers(0, n, N_SAMPLES)


def fingerprint(c):
    """Compact stand-in for an n x n fp32 cost matrix: row / column sums (fp64), diagonal, largest
    magnitude and N_SAMPLES seeded entries."""
    c = c.detach().cpu()
    n = c.shape[0]
    r, s = sample_index(n)
    d = c.double()
    return {"rowsum": d.sum(1), "colsum": d.sum(0), "diag": c.diagonal().clone(), "absmax": float(c.abs().max()),
            "samples": c[torch.from_numpy(r), torch.from_numpy(s)].clone()}


def digest(t):
    """(sha256 of the fp32 bytes, fp64 sum, fp64 sum of squares) of one state-dict tensor."""
    t = t.detach().cpu().contiguous()
    raw = t.numpy().tobytes()
    d = t.double()
    return hashlib.sha256(raw).hexdigest(), float(d.sum()), float((d * d).sum())


def objective(cost, perm):
    return float(cost.double()[torch.arange(len(perm)), perm].sum())


def run_am(ref, spec, m1, m2, loader, fixed):
    axes = [ax for pg in spec.values() for ax in pg.node]
    gm = ref.am.build_cross_module(m1, m2, axes, ref.am.cross_features_cdist)
    if fixed:
        costs = accumulate_fixed_costs(ref, spec, gm, loader, len(loader))
    else:
        costs = ref.am.compute_matching_costs(spec, gm, loader, len(loader))
    perm = {k: ref.solvers.scipy_solve_lsa(v) for k, v in costs.items()}
    return perm, costs


def gen_cfg1(ref):
    m1, m2 = make_pair("resnet18")
    spec = ref.compiler.get_permutation_spec(m1, ((1, 3, 224, 224),))
    G = {"loader": [10, 32, 224, 123]}
    loader = make_loader(*G["loader"])
    t0 = time.time()
    perm, costs = ref.am.activation_matching(spec, m1, m2, loader, num_batches=10, output_costs=True)
    G["am_seconds"] = time.time() - t0
    print(f"cfg1: reference activation_matching {G['am_seconds']:.1f}s")
    G["am/reference/perm"] = {axis_key(k): v.to(torch.int16) for k, v in perm.items()}
    G["am/reference/fingerprint"] = {axis_key(k): fingerprint(v) for k, v in costs.items()}
    G["am/reference/obj"] = {axis_key(k): objective(costs[k], perm[k]) for k in perm}
    t0 = time.time()
    model3 = ref.pm.partial_merge(spec, m1, m2, perm, costs, {k: 0.0 for k in spec})
    G["merge_seconds"] = time.time() - t0
    G["pm/r0/digest"] = {k: digest(v) for k, v in model3.state_dict().items()}
    perm_s, costs_s = run_am(ref, spec, m1, m2, loader, fixed=True)
    G["am/sum/perm"] = {axis_key(k): v.to(torch.int16) for k, v in perm_s.items()}
    G["am/sum/obj"] = {axis_key(k): objective(costs_s[k], perm_s[k]) for k in perm_s}
    G["am/sum/fingerprint"] = {axis_key(k): fingerprint(v) for k, v in costs_s.items()}
    path = os.path.join(GOLD, "cfg1_rn18_golden.pt")
    torch.save(G, path)
    print("cfg1_rn18_golden.pt:", os.path.getsize(path) // 1024, "KiB")


def gen_cfg2(ref):
    m1, m2 = make_pair("resnet50")
    spec = ref.compiler.get_permutation_spec(m1, ((1, 3, 224, 224),))
    G = {"loader": [1, 32, 224, 123]}
    loader = make_loader(*G["loader"])
    t0 = time.time()
    perm, costs = ref.am.activation_matching(spec, m1, m2, loader, num_batches=1, output_costs=True)
    G["am_seconds"] = time.time() - t0
    print(f"cfg2: reference activation_matching (one batch) {G['am_seconds']:.1f}s")
    G["am/reference/perm"] = {axis_key(k): v.to(torch.int16) for k, v in perm.items()}
    G["am/reference/obj"] = {axis_key(k): objective(costs[k], perm[k]) for k in perm}
    G["am/reference/fingerprint"] = {axis_key(k): fingerprint(v) for k, v in costs.items()}
    # how decisive each assignment is: gap between the optimum and the best single-swap alternative is
    # expensive; store the margin between the two largest entries of every row instead (diagnostic)
    G["am/reference/row_margin_min"] = {
        axis_key(k): float((v.topk(2, dim=1).values[:, 0] - v.topk(2, dim=1).values[:, 1]).min()) for k, v in costs.items()}
    path = os.path.join(GOLD, "cfg2_rn50_golden.pt")
    torch.save(G, path)
    print("cfg2_rn50_golden.pt:", os.path.getsize(path) // 1024, "KiB")


def zip_ratios(spec, budget, base):
    """get_zip_ratios (run_torchvision.py:32-54) restated on ``k.key`` (as written it calls
    ``startswith`` on Axis keys and raises, SURVEY.md 'Other quirks')."""
    layer_dict = {base[0]: 4, base[1]: 3, base[2]: 2, base[3]: 1, base[4]: 0}
    out = {}
    for k in spec:
        if k.key.startswith("layer"):
            layernum = int(k.key.split(".")[0].split("layer")[1])
            out[k] = 0.0 if layernum <= layer_dict[budget] else 1.0
        else:
            out[k] = 0.0
    return out


def gen_cfg3(ref):
    m1, m2 = make_pair("resnet50")
    spec = ref.compiler.get_permutation_spec(m1, ((1, 3, 224, 224),))
    calls = [0]

    def counting_solver(A, maximize=True):
        calls[0] += 1
        return ref.solvers.scipy_solve_lsa(A, maximize)

    t0 = time.time()
    perm, costs = ref.wm.weight_matching(spec, m1.state_dict(), m2.state_dict(), max_iter=100, seed=0,
                                         verbose=False, return_costs=True, lsa_solver=counting_solver)
    G = {"wm_seconds": time.time() - t0, "wm/lap_calls": calls[0]}
    print(f"cfg3: reference weight_matching {G['wm_seconds']:.1f}s, {calls[0]} LAP calls")
    G["wm/perm"] = {axis_key(k): v.to(torch.int16) for k, v in perm.items()}
    G["wm/fingerprint"] = {axis_key(k): fingerprint(v) for k, v in costs.items()}
    base = [1.0, 1.2, 1.55, 1.8, 2.0]  # experiments/configs/merge_configs.py:25-27 ('rn50')
    for budget in base[1:]:
        ratios = zip_ratios(spec, budget, base)
        t0 = time.time()
        model3, blocks = ref.pm.partial_merge(spec, m1, m2, perm, costs, ratios, return_blocks=True)
        tag = f"pm/{budget}"
        G[f"{tag}/seconds"] = time.time() - t0
        G[f"{tag}/ratios"] = {axis_key(k): v for k, v in ratios.items()}
        G[f"{tag}/block_sizes"] = {axis_key(k): [len(t) for t in v] for k, v in blocks.items()}
        G[f"{tag}/block_digest"] = {
            axis_key(k): [hashlib.sha256(t.cpu().numpy().astype(np.int64).tobytes()).hexdigest() for t in v]
            for k, v in blocks.items()}
        G[f"{tag}/digest"] = {k: (tuple(v.shape),) + digest(v) for k, v in model3.state_dict().items()}
        print(f"  budget {budget}: partial_merge {G[f'{tag}/seconds']:.1f}s, "
              f"{sum(v.numel() for v in model3.state_dict().values()) / 1e6:.1f} M values")
    path = os.path.join(GOLD, "cfg3_rn50_golden.pt")
    torch.save(G, path)
    print("cfg3_rn50_golden.pt:", os.path.getsize(path) // 1024, "KiB")


def bn_reset(model, loader):
    """The drivers' BN re-estimation (run_domainnet.py:327-341)."""
    model.train()
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.reset_running_stats()
    bnidx = 0
    for batch in loader:
        with torch.no_grad():
            model(batch[0].float())
        bnidx += 1
        if bnidx > 100:
            break
    model.eval()
    return model


def gen_train18(ref):
    import copy

    import torch.nn.functional as F

    RIDGES = [1e-4, 1e-6]  # relative to the mean diagonal of G; 1e-4 is the product's default (`ridge` of train)
    m1, m2 = make_pair("resnet18")
    spec = ref.compiler.get_permutation_spec(m1, ((1, 3, 224, 224),))
    G = {"am_loader": [2, 16, 224, 55], "train_loader": [41, 16, 224, 321], "max_steps": 40, "heldout": [1, 8, 224, 999],
         "ridges": RIDGES}
    perm, costs = ref.am.activation_matching(spec, m1, m2, make_loader(*G["am_loader"]), num_batches=2,
                                             output_costs=True)
    G["perm"] = {axis_key(k): v.to(torch.int16) for k, v in perm.items()}
    ratios = 0.0
    model3, blocks = ref.pm.partial_merge(spec, m1, m2, perm, costs, ratios, return_blocks=True)
    init = copy.deepcopy(model3)
    init_state = {k: v.detach().clone() for k, v in init.state_dict().items()}
    tloader = make_loader(*G["train_loader"])
    xh = make_loader(*G["heldout"])[0][0]

    t0 = time.time()
    model3 = ref.pl.train(tloader, m1, m2, model3, spec, perm, costs, ratios, False, G["max_steps"], None,
                          num_classes=1000, model_type="rn18")
    G["adam_seconds"] = time.time() - t0
    print(f"train18: reference Adam train, {G['max_steps'] + 1} batches: {G['adam_seconds']:.1f}s")
    adam_state = {k: v.detach().clone() for k, v in model3.state_dict().items()}

    # fp64 normal equations from the reference's own (X-bar, Y-bar) pairs
    perm_blocks = dict(blocks)
    for axis, pg in spec.items():
        for ax in pg.state:
            perm_blocks[ax] = perm_blocks[axis]
    a1, a2 = {}, {}
    hooks = ref.pl.capture_inputs(m1, a1) + ref.pl.capture_inputs(m2, a2)
    layers = {n: mod for n, mod in m1.named_modules() if isinstance(mod, (torch.nn.Conv2d, torch.nn.Linear))}
    acc = {}
    t0 = time.time()
    with torch.no_grad():
        for x, _ in tloader:
            m1(x)
            m2(x)
            s1, s2 = dict(a1), dict(a2)
            for name, mod in layers.items():
                X, Y = ref.pl.get_model_orig_activations(m1, m2, perm_blocks, name, s1, s2, num_classes=1000,
                                                         model_type="rn18")
                X, Y = X.double(), Y.double()
                if isinstance(mod, torch.nn.Conv2d):
                    U = F.unfold(X, mod.kernel_size, mod.dilation, mod.padding, mod.stride)
                    U = U.transpose(1, 2).reshape(-1, U.shape[1])
                    T = Y.flatten(2).transpose(1, 2).reshape(-1, Y.shape[1])
                else:
                    U, T = X, Y
                if mod.bias is not None:
                    U = torch.cat([U, torch.ones(U.shape[0], 1, dtype=U.dtype)], 1)
                d = acc.setdefault(name, {"G": 0, "R": 0, "yy": 0, "n": 0})
                d["G"] = d["G"] + U.T @ U
                d["R"] = d["R"] + U.T @ T
                d["yy"] = d["yy"] + (T * T).sum(0)
                d["n"] += T.shape[0]
    for h in hooks:
        h.remove()
    print(f"train18: fp64 normal equations {time.time() - t0:.1f}s")

    def flat_w(state, name, mod):
        W = state[f"{name}.weight"].double().flatten(1)
        if mod.bias is not None:
            W = torch.cat([W, state[f"{name}.bias"].double()[:, None]], 1)
        return W

    def loss(W, d):
        q = ((W @ d["G"]) * W).sum(1) - 2 * (W * d["R"].T).sum(1) + d["yy"]
        return float(q.sum() / (d["n"] * W.shape[0]))

    def solve_ridge(ridge):
        """fp64 ridge UPDATE of the init per layer (ratio 0: every gradient-mask entry is 1)."""
        ls_state = {k: v.clone() for k, v in init_state.items()}
        stats = {}
        for name, mod in layers.items():
            d = acc[name]
            W0, Wa = flat_w(init_state, name, mod), flat_w(adam_state, name, mod)
            A = d["G"] + ridge * float(d["G"].diagonal().mean()) * torch.eye(d["G"].shape[0], dtype=torch.float64)
            dW = torch.linalg.solve(A, d["R"] - d["G"] @ W0.T).T
            Wls = W0 + dW
            kw = Wls.shape[1] - int(mod.bias is not None)
            ls_state[f"{name}.weight"] = Wls[:, :kw].reshape(init_state[f"{name}.weight"].shape).float()
            if mod.bias is not None:
                ls_state[f"{name}.bias"] = Wls[:, kw].float()
            r, s = np.random.default_rng(7).integers(0, Wls.shape[0], 64), np.random.default_rng(8).integers(0, kw, 64)
            stats[name] = {"loss_init": loss(W0, d), "loss_adam": loss(Wa, d), "loss_lstsq": loss(Wls, d),
                           "w_norm": float(Wls.norm()), "dw_norm": float(dW.norm()),
                           "w_samples": Wls[torch.from_numpy(r), torch.from_numpy(s)].float()}
            print(f"  [ridge {ridge:g}] {name}: init {stats[name]['loss_init']:.5f} adam {stats[name]['loss_adam']:.5f} "
                  f"lstsq {stats[name]['loss_lstsq']:.5f}")
        return ls_state, stats

    def logits_of(state):
        m = copy.deepcopy(init)
        m.load_state_dict(state)
        bn_reset(m, tloader)
        with torch.no_grad():
            return m(xh).clone()

    G["logits/init"] = logits_of(init_state)
    G["logits/adam"] = logits_of(adam_state)
    # two ridges: the product default and a weak one that leaves the ill-conditioned layers (fc: 656 sample rows
    # for 513 unknowns) sensitive to fp32-level noise of the normal equations
    for ridge in G["ridges"]:
        ls_state, stats = solve_ridge(ridge)
        G[f"layer_stats/{ridge:g}"] = stats
        G[f"logits/lstsq/{ridge:g}"] = logits_of(ls_state)
    with torch.no_grad():
        G["logits/model1"], G["logits/model2"] = m1(xh).clone(), m2(xh).clone()
    rel = lambda a, b: float((a - b).norm() / b.norm())
    for ridge in RIDGES:
        print(f"train18: ridge {ridge:g}: logit rel-L2  adam vs lstsq", rel(G["logits/adam"], G[f"logits/lstsq/{ridge:g}"]),
              " init vs lstsq", rel(G["logits/init"], G[f"logits/lstsq/{ridge:g}"]))
    print("train18: lstsq 1e-4 vs 1e-6", rel(G["logits/lstsq/0.0001"], G["logits/lstsq/1e-06"]))
    path = os.path.join(GOLD, "train18_golden.pt")
    torch.save(G, path)
    print("train18_golden.pt:", os.path.getsize(path) // 1024, "KiB")


def main():
    if os.environ.get("PYTHONHASHSEED") != "0":
        sys.exit("run with PYTHONHASHSEED=0 (pins the reference's set iteration order)")
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    ref = load_reference()
    which = sys.argv[1:] or ["cfg2", "cfg3", "cfg1", "train18"]
    for name in which:
        {"cfg1": gen_cfg1, "cfg2": gen_cfg2, "cfg3": gen_cfg3, "train18": gen_train18}[name](ref)


if __name__ == "__main__":
    main()
