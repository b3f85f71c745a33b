"""CPU-side tests (no GPU): the C-ABI library loads and exports every declared symbol, the
spec compiler reproduces the reference's specs, the data model interoperates with the
reference's, and the multi-GPU plumbing works across two gloo ranks."""
import ctypes
import json
import os
import re
import subprocess
import sys

import pytest
import torch

from conftest import GOLDEN, ROOT, load_spec_json


def test_cabi_library_exports_every_declared_symbol():
    from pleas_merging_b200 import _native, build

    path = build.build()
    lib = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, "include", "pleas_b200.h")).read()
    declared = set(re.findall(r"\b(plb_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_native.EXPORTED_SYMBOLS), declared ^ set(_native.EXPORTED_SYMBOLS)
    for sym in declared:
        assert hasattr(lib, sym), sym
    lib.plb_version.restype = ctypes.c_int
    assert lib.plb_version() >= 100
    # host-only helper: plane geometry
    lib.plb_plane_bytes.restype = ctypes.c_int64
    lib.plb_plane_bytes.argtypes = [ctypes.c_int64, ctypes.c_int64, ctypes.POINTER(ctypes.c_int32),
                                    ctypes.POINTER(ctypes.c_int32)]
    rg, kb = ctypes.c_int32(), ctypes.c_int32()
    assert lib.plb_plane_bytes(200, 1000, ctypes.byref(rg), ctypes.byref(kb)) == 25 * 63 * 512
    assert (rg.value, kb.value) == (25, 63)  # ceil(200/8) row groups, ceil(1000/16) k-blocks, 512-B panels
    assert lib.plb_plane_bytes(0, 5, None, None) < 0  # invalid argument, no crash


def test_gemm_problem_struct_matches_header():
    from pleas_merging_b200 import _native

    assert ctypes.sizeof(_native.GemmProblem) == 5 * 8 + 8 * 4


def test_product_fails_loudly_without_cuda():
    """No CPU fallback: calling an operator on CPU tensors raises instead of computing."""
    import pleas_merging_b200 as P

    with pytest.raises(TypeError):
        P.cross_features_cdist(torch.randn(2, 4, 3, 3), torch.randn(2, 4, 3, 3), 1)
    if not torch.cuda.is_available():
        from oracle import tinynet

        m1, m2 = tinynet.make_pair()
        spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
        with pytest.raises(RuntimeError):
            P.activation_matching(spec, m1, m2, tinynet.make_loader(1, 2), 1)


def test_missing_library_raises(monkeypatch, tmp_path):
    from pleas_merging_b200 import _native

    monkeypatch.setattr(_native, "_lib", None)
    monkeypatch.setattr(_native, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _native.lib()


def _spec_json(spec):
    return [{"key": [k.key, k.axis], "size": pg.size, "state": sorted([a.key, a.axis] for a in pg.state),
             "node": sorted([a.key, a.axis] for a in pg.node)} for k, pg in spec.items()]


@pytest.mark.parametrize("name", ["tiny", "resnet18", "resnet50", "resnet50_nofc", "resnet101"])
def test_permutation_spec_equals_reference(name):
    import torchvision

    import pleas_merging_b200 as P
    from oracle import tinynet

    torch.manual_seed(0)
    if name == "tiny":
        model, shape = tinynet.TinyResNet(12, 10).eval(), (1, 3, 16, 16)
    else:
        model = getattr(torchvision.models, name.replace("_nofc", ""))().eval()
        if name.endswith("_nofc"):
            model.fc = torch.nn.Identity()
        shape = (1, 3, 64, 64)
    spec = P.get_permutation_spec(model, (shape,))
    with open(os.path.join(GOLDEN, f"spec_{name}.json")) as f:
        assert _spec_json(spec) == json.load(f)  # keys, order, sizes, state and node sets


def test_spec_invariance_selfcheck():
    import pleas_merging_b200 as P
    from oracle import tinynet

    m, _ = tinynet.make_pair()
    spec = P.get_permutation_spec(m, ((1, 3, 16, 16),))
    assert P.check_permutation_spec(m, spec, torch.randn(2, 3, 16, 16)) == set()


def test_compiler_rejects_unknown_ops():
    import pleas_merging_b200 as P

    class Odd(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.l = torch.nn.Linear(4, 4)

        def forward(self, x):
            return torch.fft.fft(self.l(x)).real

    with pytest.raises(NotImplementedError):
        P.get_permutation_spec(Odd(), ((2, 4),))


def test_axis_interoperates_with_reference_dataclass():
    """Dicts keyed by the reference's frozen-dataclass Axis can be indexed with ours and vice versa."""
    from dataclasses import dataclass

    import pleas_merging_b200 as P

    @dataclass(frozen=True)
    class RefAxis:  # same definition as pleas/core/utils.py:16-31
        key: str
        axis: int

    ours, theirs = P.Axis("layer1.0.conv1.weight", 0), RefAxis("layer1.0.conv1.weight", 0)
    assert hash(ours) == hash(theirs) and ours == theirs and theirs == ours
    assert {theirs: 1}[ours] == 1 and {ours: 2}[theirs] == 2
    assert ours != P.Axis("layer1.0.conv1.weight", 1) and str(ours) == "layer1.0.conv1.weight:0"
    assert P.Axis(*ours) == ours


def test_perm_helpers_and_apply_perm_cpu():
    import pleas_merging_b200 as P
    from oracle import ref_oracle as O
    from oracle import tinynet

    m, _ = tinynet.make_pair()
    spec = P.get_permutation_spec(m, ((1, 3, 16, 16),))
    perm = P.make_random_perm(spec, generator=torch.Generator().manual_seed(0))
    inv = P.invert_perm(perm)
    assert all(torch.equal(perm[k][inv[k]], torch.arange(len(perm[k]))) for k in perm)
    assert P.perm_eq(perm, {k: v.clone() for k, v in perm.items()}) and not P.perm_eq(perm, inv)
    sd = P.apply_perm(perm, spec, m.state_dict())
    jspec = load_spec_json("tiny")
    ref = {k: v.numpy().copy() for k, v in m.state_dict().items() if v.dim() > 0}
    for g in jspec:
        O.apply_perm_group(g, perm[P.Axis(*g["key"])].numpy(), ref)
    for k, v in ref.items():
        assert (sd[k].numpy() == v).all(), k


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from pleas_merging_b200 import parallel
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[2]}", rank=int(sys.argv[3]), world_size=2)
rank, world = parallel.world()
loader = [(torch.full((2, 2), float(i)), 0) for i in range(7)]
for mode in ("sum", "reference"):
    sh = parallel.BatchSharder(loader, 5)            # 5 of the 7 batches, dealt round-robin
    flat = torch.zeros(4)
    seen = []
    for idx, (x, _) in sh:
        seen.append(idx)
        if mode == "reference":
            flat.zero_()
        flat += x.flatten()
    assert seen == list(range(rank, 5, 2)), seen
    assert sh.total == 5 and sh.owns_last() == (rank == 0)   # batch 4 belongs to rank 0
    parallel.combine_costs_(flat, sh, mode)
    want = float(sum(range(5))) if mode == "sum" else 4.0
    assert torch.equal(flat, torch.full((4,), want)), (mode, flat)
# layer-parallel solves: owners get the sum of their segments, then a flat all-reduce shares results
costs = [5.0, 1.0, 4.0, 2.0, 2.0]
owners = parallel.assign_owners(costs, world)
assert owners == [0, 1, 1, 1, 0], owners            # LPT greedy: 5->r0, 4->r1, 2->r1, 2->r0, 1->r1
lens = [3, 2, 4, 1, 2]
order = [i for r in range(world) for i in range(5) if owners[i] == r]   # buffer laid out owner by owner
segs, off = {}, 0
for i in order:
    segs[i] = (off, lens[i]); off += lens[i]
flat = torch.arange(off, dtype=torch.float64) * (rank + 1)
parallel.reduce_to_owners_(flat, [segs[i] for i in order], [owners[i] for i in order])
out = torch.zeros(off, dtype=torch.float64)
for i in order:
    lo, n = segs[i]
    if owners[i] == rank:
        assert torch.equal(flat[lo:lo + n], torch.arange(lo, lo + n, dtype=torch.float64) * 3), (i, flat)
        out[lo:lo + n] = flat[lo:lo + n] * 2            # the owner's "solve"
parallel.allreduce_sum_(out)
assert torch.equal(out, torch.arange(off, dtype=torch.float64) * 6), out
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_two_rank_sharding_and_allreduce_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(port), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"ok {r}" in o, o


def test_assign_owners_balances_resnet50_solves():
    """Layer-parallel PLeaS: the LPT deal keeps the heaviest rank within 10 % of the mean for
    the ResNet-50 layer mix (K^3/3 + K^2 Co per layer) — or at the single heaviest layer (the
    three K=4608 convolutions of layer4 are 23 % of the work each) once that exceeds the mean."""
    from pleas_merging_b200.parallel import assign_owners

    widths = [(64, 3), (128, 4), (256, 6), (512, 3)]
    layers, cin = [(3 * 49, 64)], 64
    for w, blocks in widths:
        for b in range(blocks):
            layers += [(cin, w), (w * 9, w), (w, 4 * w)] + ([(cin, 4 * w)] if b == 0 else [])
            cin = 4 * w
    layers.append((2049, 1000))
    costs = [k ** 3 / 3.0 + k * k * co for k, co in layers]
    assert len(costs) == 54
    for world in (1, 2, 4, 8):
        owners = assign_owners(costs, world)
        load = [sum(c for c, o in zip(costs, owners) if o == r) for r in range(world)]
        assert max(load) <= max(1.10 * sum(costs) / world, max(costs)), (world, load)
        assert owners == assign_owners(costs, world)


@pytest.mark.parametrize("name", ["tiny", "resnet18", "resnet50"])
def test_flop_accounting_equals_reference(name):
    """count_linear_flops / partial_merge_flops against values produced by the unmodified reference
    (tests/golden/budget_golden.json; pleas/core/utils.py:558-617, partial_matching.py:205-226)."""
    import torchvision

    import pleas_merging_b200 as P
    from oracle import tinynet
    from pleas_merging_b200.methods.budget import count_linear_flops, partial_merge_flops

    with open(os.path.join(GOLDEN, "budget_golden.json")) as f:
        gold = json.load(f)[name]
    torch.manual_seed(0)
    if name == "tiny":
        m, shape = tinynet.TinyResNet(12, 10).eval(), (1, 3, 16, 16)
    else:
        m, shape = getattr(torchvision.models, name)().eval(), (1, 3, 64, 64)
    spec = P.get_permutation_spec(m, (shape,))
    flops, terms = count_linear_flops(spec, m, (shape,))
    assert int(flops) == gold["flops"]
    assert [[int(c)] + [[a.key, a.axis] for a in axes] for c, *axes in terms] == gold["terms"]
    mixed = {P.Axis(k, a): r for k, a, r in gold["mixed_ratios"]}
    for cn, r in (("r0", 0.0), ("r1", 1.0), ("r03", 0.3), ("mixed", mixed)):
        assert partial_merge_flops(spec, terms, r) == pytest.approx(gold["merge_flops"][cn], rel=1e-12), cn
    assert partial_merge_flops(spec, terms, 0.0) == pytest.approx(flops, rel=1e-12)


def test_zip_ratios_rule():
    import torchvision

    import pleas_merging_b200 as P
    from pleas_merging_b200.methods.budget import get_zip_ratios

    spec = P.get_permutation_spec(torchvision.models.resnet18().eval(), ((1, 3, 64, 64),))
    base = [1.0, 1.24, 1.46, 1.71, 2.0]  # experiments/configs/merge_configs.py:25 (rn18)
    assert set(get_zip_ratios(spec, 1.0, base).values()) == {0.0}
    r = get_zip_ratios(spec, 1.46, base)  # layers 1-2 merged, 3-4 separate, stem merged
    for k, v in r.items():
        want = 1.0 if k.key.startswith(("layer3", "layer4")) else 0.0
        assert v == want, k
    r2 = get_zip_ratios(spec, 2.0, base)
    assert all((v == 1.0) == k.key.startswith("layer") for k, v in r2.items())


def test_mask_classes_equal_unique_rows_of_the_reference_mask():
    """_LayerLS.mask_classes (analytic row classes) == torch.unique over the materialised gradient
    mask (reference index order, pleas_merging.py:52-59) for merged / partially merged layers."""
    import importlib

    PM = importlib.import_module("pleas_merging_b200.methods.pleas_merging")
    e = lambda n: torch.zeros(n, dtype=torch.int64)
    cases = [((12, 8, 3, 3), (8, 0), (12, 0), False), ((14, 10, 3, 3), (6, 2), (8, 3), False),
             ((10, 9), (5, 2), (6, 2), True), ((9, 20, 1, 1), (8, 6), (5, 2), True),
             ((16, 12, 1, 1), (6, 3), (16, 0), False), ((7, 3, 7, 7), (3, 0), (5, 1), False)]
    for wshape, (ni, mi), (no, mo), bias in cases:
        a = object.__new__(PM._LayerLS)
        a.bi, a.bo, a.has_bias = (e(ni), e(ni), e(mi), e(mi)), (e(no), e(no), e(mo), e(mo)), bias
        mask = a.mask2d(wshape)
        pats, inv = a.mask_classes(wshape)
        assert pats.shape[1] == mask.shape[1] and inv.shape[0] == mask.shape[0]
        assert torch.equal(pats[inv], mask), (wshape, ni, mi, no, mo)
        assert pats.shape[0] == torch.unique(mask, dim=0).shape[0]


@pytest.mark.parametrize("name", ["r0", "r05", "r1", "mixed"])
def test_permute_final_features_equals_reference(eval_golden, name):
    """permute_final_features is device-agnostic: on the reference's own fc blocks and features it
    returns the reference's tensors bit for bit (pleas_merging.py:436-465)."""
    from pleas_merging_b200.methods.evaluation import permute_final_features

    fc_perm, feats = eval_golden[f"{name}/fc_perm"], eval_golden[f"{name}/features"]
    for idx in (0, 1):
        out = permute_final_features(feats, fc_perm, idx)
        assert torch.equal(out, eval_golden[f"{name}/out{idx}"])


def test_qp_ratios_feasible_and_near_optimal():
    """qp_ratios (SURVEY 8f n2; reference partial_matching.py:229-257 needs Gurobi, so no golden
    exists): the result meets the FLOP budget, uses it up, and its objective is within 1 % of the
    best of SciPy SLSQP multi-starts (test-only checker) on ResNet-18 terms; on a two-group toy it
    matches a brute-force grid."""
    import numpy as np
    import torchvision
    from scipy.optimize import minimize

    import pleas_merging_b200 as P
    from pleas_merging_b200.methods.budget import count_linear_flops, partial_merge_flops, qp_ratios

    m = torchvision.models.resnet18().eval()
    spec = P.get_permutation_spec(m, ((1, 3, 64, 64),))
    _, terms = count_linear_flops(spec, m, ((1, 3, 64, 64),))
    keys = list(spec.keys())
    rng = np.random.default_rng(0)
    base = partial_merge_flops(spec, terms, 0.0)
    for budget in (1.2, 1.55, 1.8):
        w = {k: float(x) for k, x in zip(keys, rng.uniform(-0.2, 1.0, len(keys)))}
        out = qp_ratios(spec, terms, budget, w)
        assert set(out) == {k.key for k in keys} and all(0.0 <= v <= 1.0 for v in out.values())
        r = {k: out[k.key] for k in keys}
        used = partial_merge_flops(spec, terms, r) / base
        assert used <= budget * (1 + 1e-9) and used >= budget * 0.999, (budget, used)
        wv = np.array([max(w[k], 1e-5) for k in keys])
        val = float(sum(wv[i] * r[k] for i, k in enumerate(keys)))
        fun = lambda x: partial_merge_flops(spec, terms, {k: float(v) for k, v in zip(keys, x)}) / base
        best = 0.0
        for s in range(4):
            x0 = rng.uniform(0, 1, len(keys)) * (0.0 if s == 0 else 1.0)
            res = minimize(lambda x: -float(wv @ x), x0, method="SLSQP", bounds=[(0, 1)] * len(keys),
                           constraints=[{"type": "ineq", "fun": lambda x: budget - fun(x)}], options={"maxiter": 300})
            if res.success and fun(res.x) <= budget * (1 + 1e-6):
                best = max(best, float(wv @ res.x))
        assert val >= 0.99 * best, (budget, val, best)
    # extremes
    assert all(v == 1.0 for v in qp_ratios(spec, terms, 2.5, {k: 1.0 for k in keys}).values())
    assert all(v == 0.0 for v in qp_ratios(spec, terms, 1.0, {k: 1.0 for k in keys}).values())


@pytest.mark.parametrize("name", ["r05", "r025", "mixed"])
def test_weight_matching_partial_equals_reference(name):
    """SURVEY 8f n4: weight_matching_partial / apply_perm_with_padding / remove_zero_block
    (partial_matching.py:260-463) reproduce the reference's permutation and BOTH rewritten state
    dicts on the tiny pair.  The host logic is device-agnostic, so it runs here with CPU plug-ins in
    the two operator slots (the oracle's SciPy-identical LAP and a torch matmul); the product
    defaults are the library's GPU LAP and tcgen05 Gram."""
    import numpy as np

    import pleas_merging_b200 as P
    from oracle import ref_oracle as O
    from oracle import tinynet
    from pleas_merging_b200.methods.weight_matching_partial import weight_matching_partial

    G = torch.load(os.path.join(ROOT, "tests", "golden", "wmp_golden.pt"), weights_only=False)

    def cpu_lsa(A, maximize=True):
        return torch.from_numpy(np.asarray(O.solve_lsa(A.numpy(), maximize)[0], dtype=np.int64))

    def cpu_cross(x, y, a):
        x = torch.movedim(x, a, 0).reshape(x.shape[a], -1)
        y = torch.movedim(y, a, 0).reshape(y.shape[a], -1)
        return x @ y.T

    m1, m2 = tinynet.make_pair(12, 10)
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    ratios = {k: G[f"{name}/ratios"][f"{k.key}:{k.axis}"] for k in spec}
    sa = {k: v.clone() for k, v in m1.state_dict().items()}
    sb = {k: v.clone() for k, v in m2.state_dict().items()}
    perm = weight_matching_partial(spec, sa, sb, ratios, max_iter=20, inplace=True, verbose=False, seed=0,
                                   lsa_solver=cpu_lsa, cross_weights=cpu_cross)
    for k in spec:
        assert torch.equal(perm[k], G[f"{name}/perm"][f"{k.key}:{k.axis}"]), k
    for tag, mine in (("state_a", sa), ("state_b", sb)):
        gold = G[f"{name}/{tag}"]
        assert set(mine) == set(gold)
        for k, v in gold.items():
            assert mine[k].shape == v.shape and torch.equal(mine[k], v), (tag, k)


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU path timed beside the B200 arm) runs without a GPU and
    prints exactly one JSON line carrying the contract's keys (small model / sample here)."""
    import json

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "resnet18",
                          "--steps", "1", "--warmup", "0", "--cpu-sample", "2"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["unit"] == "samples/s"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_bench_reference_arm_dumps_the_timed_batches_costs(tmp_path):
    """`bench.py --impl reference --dump-outputs DIR` writes one float32 cost matrix per permutation group: the
    -cdist sums over the `--steps` timed batches alone (the warm-up batch excluded), recomputed here from the
    benchmark's seeded inputs (torch CPU generator 123, `--cpu-sample` samples of 224x224 per batch)."""
    import numpy as np

    import bench
    from oracle import ref_oracle as O

    steps, warm, b = 2, 1, 2
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "resnet18",
                          "--steps", str(steps), "--warmup", str(warm), "--cpu-sample", str(b),
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
    spec = load_spec_json("resnet18")
    m1, m2 = bench.make_models("resnet18")
    g = torch.Generator().manual_seed(123)
    loader = [(torch.randn(b, 3, 224, 224, generator=g), 0) for _ in range(warm + steps)]
    want = O.matching_costs(spec, m1, m2, loader[warm:], steps, "cdist", "sum")
    assert sorted(f.name for f in tmp_path.iterdir()) == sorted(f"cost_{k}_{a}.npy" for k, a in want)
    for (key, axis), c in want.items():
        got = np.load(tmp_path / f"cost_{key}_{axis}.npy")
        assert got.dtype == np.float32 and got.shape == c.shape, key
        # same computation; only the host thread count may differ between the two processes
        assert np.abs(got.astype(np.float64) - c).max() <= 1e-5 * np.abs(c).max(), key


def test_built_library_is_sm100a_native_sass():
    """The in-tree library really is tcgen05 / TMA / redux code for sm_100a (cuobjdump -sass, no GPU
    needed): UTCHMMA + LDTM (TMEM loads) + UBLKCP (bulk copies) in the GEMM, UTCHMMA + LDGSTS in the
    fused narrow-tap kernel, REDUX in the LAP kernel — and the MMAs of a k-block are issued back to
    back from uniform registers (no per-MMA ELECT/R2UR uniformisation loop)."""
    import shutil

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from pleas_merging_b200 import build

    lib = build.build()
    sass = subprocess.run([cuobjdump, "-sass", lib], capture_output=True, text=True, timeout=300).stdout
    assert "sm_100a" in sass
    funcs = {}
    name = None
    for line in sass.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
            funcs[name] = []
        elif name is not None:
            funcs[name].append(line)

    def body(sub):
        hits = [n for n in funcs if sub in n]
        assert hits, sub
        return {n: "\n".join(funcs[n]) for n in hits}

    for n, b in body("gemm3xtf32_v2_kernel").items():
        assert "UTCHMMA" in b and "LDTM" in b and "UBLKCP" in b and "UTCBAR" in b, n
        assert b.count("BRA.U.ANY") <= 6, (n, b.count("BRA.U.ANY"))  # was 24 with the lane == 0 guard
    for n, b in body("gram_direct_kernel").items():
        assert "UTCHMMA" in b and "LDTM" in b and "LDGSTS" in b, n
    assert all("REDUX" in b for b in body("lap_kernel_v2").values())
    # v3 (product path): warp arg-min by redux, and the shared window base is not re-derived per step
    # (at most the handful of S2R/S2UR SR_CgaCtaId outside the step loop)
    for n, b in body("lap_kernel_v3").items():
        assert "REDUX" in b, n
        if "ILi1E" in n or "ILi2E" in n:  # every group of a ResNet pair (n <= 2048)
            assert "STL" not in b and "LDL" not in b, n  # column state stays in registers
    # round 2: the TMA-fed Gram kernel — tensor-map loads (UTMALDG), TMEM loads, and for the CTA-pair
    # instantiation 2-CTA MMAs with a multicast commit
    tma = body("gram_tma_kernel")
    assert len(tma) >= 6
    for n, b in tma.items():
        assert "UTMALDG" in b and "UTCHMMA" in b and "LDTM" in b, n
        if "ILi1E" in n:  # stage hand-overs use CTA-scope barrier semantics: no GPU-scope fence anywhere
            assert "MEMBAR.ALL.GPU" not in b and "CCTL.IVALL" not in b, n
    pair = [b for n, b in tma.items() if "ILi2E" in n]
    assert pair and all("UTCHMMA.2CTA" in b and "UTCBAR.2CTA.MULTICAST" in b for b in pair)


def test_conv_kernel_sass_and_packed_geometry():
    """The convolution kernel (csrc/conv.cu) is what its header says: tensor-map TMA for the weights (UTMALDG),
    4-byte cp.async gathers (zero padding = ignore-src copies) for the activations (LDGSTS), the A operand written to tensor
    memory (STTM) and MMAs that take it from there (UTCHMMA with a tmem A operand), packed f32x2 promotion adds in
    the production instantiation; and the packed-weight size helper (host-only) follows include/pleas_b200.h."""
    import ctypes
    import shutil

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from pleas_merging_b200 import _native, build

    lib = build.build()
    sass = subprocess.run([cuobjdump, "-sass", lib], capture_output=True, text=True, timeout=300).stdout
    bodies, name = {}, None
    for line in sass.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
            bodies[name] = []
        elif name is not None:
            bodies[name].append(line)
    conv = {n: "\n".join(b) for n, b in bodies.items() if "conv3xtf32_kernel" in n}
    assert len(conv) >= 4  # TN 64 / 128 x production / experiments builds
    for n, b in conv.items():
        assert "UTMALDG" in b and "STTM" in b and "LDTM" in b and "LDGSTS" in b, n
        mma = [l for l in b.splitlines() if "UTCHMMA" in l]
        assert len(mma) >= 12 and all(l.split("UTCHMMA")[1].strip().startswith("tmem[") for l in mma), n
        assert "MEMBAR.ALL.GPU" not in b, n
    assert any("FADD2" in b for b in conv.values())
    h = _native.lib()
    # channel-block form: [2][KH*KW][Cout][Cin]
    assert h.plb_conv_packed_floats(256, 128, 3, 3) == 2 * 9 * 256 * 128
    # flat form (Cin % 32 != 0): kernel rows padded to 8 taps, K = 3*7*8 = 168 -> 192
    assert h.plb_conv_packed_floats(64, 3, 7, 7) == 2 * 64 * 192
    assert h.plb_conv_packed_floats(0, 3, 7, 7) == 0
    import torch
    from pleas_merging_b200 import conv as C

    assert not C.eligible(torch.nn.Conv2d(64, 64, 3))            # CPU weights: the module keeps its own forward
    assert not C.eligible(torch.nn.Conv2d(64, 64, 3, groups=2))


def test_parallel_helpers_single_process_edges():
    """No process group: the collectives are no-ops, every item belongs to rank 0, and a sharder
    over an empty / short loader yields what exists."""
    from pleas_merging_b200 import parallel

    assert parallel.world() == (0, 1)
    assert parallel.assign_owners([], 4) == []
    assert parallel.assign_owners([3.0, 1.0, 2.0], 1) == [0, 0, 0]
    assert parallel.assign_owners([1.0, 1.0, 1.0, 1.0], 4) == [0, 1, 2, 3]  # ties: lowest rank, input order
    flat = torch.arange(6.0)
    assert parallel.reduce_to_owners_(flat, [(0, 3), (3, 3)], [0, 0]) is flat and torch.equal(flat, torch.arange(6.0))
    assert parallel.allreduce_sum_(flat) is flat
    sh = parallel.BatchSharder([], 5)
    assert list(sh) == [] and sh.total == 0 and not sh.owns_last()
    sh = parallel.BatchSharder([(torch.zeros(1), 0)] * 2, 5)  # loader shorter than num_batches
    assert [i for i, _ in sh] == [0, 1] and sh.total == 2 and sh.owns_last()
    sh = parallel.BatchSharder([(torch.zeros(1), 0)] * 7, 5, rank=1, world_size=2)
    assert [i for i, _ in sh] == [1, 3] and sh.total == 5 and not sh.owns_last()


def test_public_api_signatures_match_the_reference():
    """Drop-in contract: every public function of the reference on the merge path exists here with
    the same positional parameter names in the same order and the same plain default values
    (tests/golden/api_signatures.json, generated from the unmodified reference); this package may
    only ADD keyword parameters after them."""
    import inspect
    import json

    import pleas_merging_b200 as P
    from pleas_merging_b200 import methods as M
    from pleas_merging_b200.core import solvers, utils

    with open(os.path.join(ROOT, "tests", "golden", "api_signatures.json")) as f:
        gold = json.load(f)
    assert len(gold) >= 25
    for name, params in gold.items():
        fn = next((getattr(m, name) for m in (M, P, solvers, utils) if hasattr(m, name)), None)
        assert fn is not None, f"{name} is missing"
        mine = list(inspect.signature(fn).parameters.values())
        assert [p.name for p in mine[:len(params)]] == [a for a, _ in params], name
        for prm, (_, default) in zip(mine, params):
            if default == "<required>":
                assert prm.default is inspect.Parameter.empty, (name, prm.name)
            elif default == "<callable>":
                assert callable(prm.default), (name, prm.name)
            else:
                got = list(prm.default) if isinstance(prm.default, tuple) else prm.default
                assert got == default, (name, prm.name, got, default)
        for extra in mine[len(params):]:  # additions must not break positional calls written for the reference
            assert extra.default is not inspect.Parameter.empty or extra.kind is extra.KEYWORD_ONLY, (name, extra.name)


def test_tma_planning_helpers_and_struct_mirrors():
    """Host-side planning of the TMA-fed Gram kernel and of the grouped epilogue (no compute calls):
    tiling from the C ABI's geometry helper, K-split choice, block counts, ctypes mirrors of the header structs."""
    import ctypes

    from pleas_merging_b200 import _native, ops

    assert ops.tma_geometry(64) == (1, 1, 1, 128, 64)
    assert ops.tma_geometry(128) == (1, 1, 1, 128, 128)
    assert ops.tma_geometry(256) == (2, 1, 1, 256, 256)
    assert ops.tma_geometry(320) == (2, 2, 2, 512, 512)  # rows past 320 are TMA zero fill
    assert ops.tma_geometry(2048) == (2, 8, 8, 2048, 2048)
    # K splits: one narrow tile spreads over (almost) all SMs; 16 wide tiles take few splits; never more splits
    # than a quarter of the boxes
    assert 100 <= ops.choose_tma_splits(1, 1, 12544, 128 * 64, 148) <= 148
    assert ops.choose_tma_splits(16, 2, 224, 256 * 256, 148) in (4, 5, 9)
    assert ops.choose_tma_splits(1, 2, 8, 256 * 256, 148) <= 2
    assert ops.choose_tma_splits(4, 2, 3, 256 * 256, 148) == 1
    # grouped epilogue: 256-column x 16-row tiles from 256 units up, 64 x 64 below
    assert ops.finalize_grouped_blocks(64) == 1 and ops.finalize_grouped_blocks(65) == 4
    assert ops.finalize_grouped_blocks(256) == 16 and ops.finalize_grouped_blocks(2048) == 8 * 128
    assert ctypes.sizeof(_native.FinalizeTap) == 80 and ctypes.sizeof(_native.FinalizeGroup) == 32
    header = open(os.path.join(ROOT, "include", "pleas_b200.h")).read()
    for field in ("partial", "qa", "qb", "sa", "sb", "ld_m", "ld_n", "K", "splits", "n_affine", "affine"):
        assert re.search(r"typedef struct PlbFinalizeTap \{[^}]*\b%s\b" % field, header, re.S), field
    for field in ("cost", "ldc", "n", "tap_begin", "tap_end", "block_begin"):
        assert re.search(r"typedef struct PlbFinalizeGroup \{[^}]*\b%s\b" % field, header, re.S), field


def test_runner_cache_fingerprints_detect_what_invalidates_a_captured_graph():
    """The calibration runner (fx graph + plans + CUDA graph) is reused across activation_matching calls only
    while every parameter / buffer keeps its storage, shape and dtype and the modules keep their training flags."""
    import importlib

    import torch

    from oracle import tinynet

    AM = importlib.import_module("pleas_merging_b200.methods.activation_matching")
    import pleas_merging_b200 as P

    m, _ = tinynet.make_pair(12, 10)
    fp = AM._model_fingerprint(m)
    assert AM._model_fingerprint(m) == fp
    with torch.no_grad():
        next(m.parameters()).add_(1.0)  # new VALUES in the same storage: a replay reads them in place
    assert AM._model_fingerprint(m) == fp
    m.train()
    assert AM._model_fingerprint(m) != fp  # BatchNorm would run with batch statistics
    m.eval()
    assert AM._model_fingerprint(m) == fp
    first = next(m.parameters())
    first.data = first.data.clone()  # re-allocated storage: a captured graph would read the old one
    assert AM._model_fingerprint(m) != fp
    spec = P.get_permutation_spec(m, ((1, 3, 16, 16),))
    assert AM._spec_fingerprint(spec) == AM._spec_fingerprint(P.get_permutation_spec(m, ((1, 3, 16, 16),)))


def test_batchnorm_derivation_bound():
    """BN_AFFINE_MAX_GROWTH admits a derived BatchNorm tap while max(kappa / kappa') of one model times the other's
    stays within the bound: kappa^2 = 1 + mean^2 / (var + eps) of the convolution output, kappa'^2 = 1 + beta^2 /
    gamma^2 of the BatchNorm output."""
    import importlib

    AM = importlib.import_module("pleas_merging_b200.methods.activation_matching")

    def bn(mean, var, gamma, beta, affine=True):
        m = torch.nn.BatchNorm2d(len(mean), affine=affine, eps=0.0).eval()
        m.running_mean.copy_(torch.tensor(mean))
        m.running_var.copy_(torch.tensor(var))
        if affine:
            m.weight.data.copy_(torch.tensor(gamma))
            m.bias.data.copy_(torch.tensor(beta))
        return m

    def growth(m):
        return AM.affine_growth(m.running_mean, m.running_var, m.eps, m.weight, m.bias)

    fresh = torch.nn.BatchNorm2d(64).eval()  # random init: mean 0, var 1, gamma 1, beta 0
    assert growth(fresh) == 1.0 and AM._bn_derivable(fresh, fresh)
    assert AM.BN_AFFINE_MAX_GROWTH >= 1.0
    assert growth(bn([3.0, 0.0], [1.0, 4.0], [1.0, 1.0], [0.0, 0.0])) == pytest.approx(10 ** 0.5)   # worst unit
    assert growth(bn([3.0], [1.0], [2.0], [6.0])) == pytest.approx(1.0)                             # beta/gamma = mean/sd
    assert growth(bn([0.0], [1.0], [-1.0], [1.0])) == pytest.approx(0.5 ** 0.5)                      # sign of gamma
    assert growth(bn([5.0], [1.0], [0.0], [1.0])) == 0.0             # gamma = 0: a constant output, derived exactly
    assert growth(bn([2.0], [4.0], None, None, affine=False)) == pytest.approx(2 ** 0.5)
    assert not AM._bn_derivable(bn([float("nan")], [1.0], [1.0], [0.0]), fresh)
    b = AM.BN_AFFINE_MAX_GROWTH
    edge = bn([(b - 1.0) ** 0.5], [1.0], [1.0], [0.0])                # kappa = sqrt(b) on both sides
    assert AM._bn_derivable(edge, edge)
    worse = bn([(1.01 * b - 1.0) ** 0.5], [1.0], [1.0], [0.0])
    assert not AM._bn_derivable(worse, worse)
    assert AM._bn_derivable(worse, bn([0.0], [1.0], [1.0], [1.0]))   # the other model's kappa' = sqrt(2) makes room

    from oracle import tinynet

    m1, m2 = tinynet.make_pair(12, 10)  # perturbed statistics around mean 0, var 1: every BatchNorm stays derived
    for (_, a), (_, c) in zip(((n, m) for n, m in m1.named_modules() if isinstance(m, torch.nn.BatchNorm2d)),
                              ((n, m) for n, m in m2.named_modules() if isinstance(m, torch.nn.BatchNorm2d))):
        assert AM._bn_derivable(a, c)
