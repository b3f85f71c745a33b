"""The 3xTF32 tcgen05 convolution (csrc/conv.cu, plb_conv2d_forward) against the fp64 convolution of the same
inputs, through the C ABI: every geometry class of the ResNet family the configs use (1x1, 3x3 pad 1, strided, the
3-channel 7x7 stem, 7x7 / 14x14 maps whose rows are not 16-byte multiples, ragged position / channel tiles, bias),
and the edges of what ``conv.eligible()`` admits beyond it: non-square kernels, asymmetric and oversized padding,
strides larger than the kernel, every flat-form row width, the flat-K limit, odd box counts, every output-channel
tile shape, inputs of more than 2^31 elements.

Two bars, both against fp64:
  * global: max|y - y64| <= 3e-6 max|y64| (fp32 cuDNN itself sits at ~1e-6);
  * elementwise: |y - y64| <= TOL * B with B = conv(|x|, |w|) + |bias|, the condition bound of each output, so an
    error confined to small outputs (borders, ragged tails, low-magnitude channels) cannot hide under the largest.
"""
import ctypes

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# Elementwise bar, relative to the condition bound B.  Measured over every case of this file on a B200 (1000 W power
# limit): max |y - y64| / B = 2.9e-7 for the convolution outputs, 5.8e-7 for the fused BatchNorm outputs (relative to
# |s| B, after the 2^-24 |t| allowance).  TOL leaves a margin of 3.4x and 1.7x over them; a kernel that drops one of
# the three products reaches 4e-4.
TOL = 1e-6
GLOBAL_TOL = 3e-6
PLB_ESIZE = -2

CASES = [
    # (NB, Cin, H, W, Cout, (KH, KW), stride, (pad_h, pad_w), bias)
    # the ResNet family
    (2, 64, 56, 56, 64, (1, 1), 1, (0, 0), False),
    (2, 64, 56, 56, 256, (1, 1), 1, (0, 0), False),
    (3, 64, 28, 28, 64, (3, 3), 1, (1, 1), False),
    (2, 128, 56, 56, 128, (3, 3), 2, (1, 1), False),
    (2, 256, 56, 56, 512, (1, 1), 2, (0, 0), False),
    (5, 256, 14, 14, 256, (3, 3), 1, (1, 1), True),
    (32, 512, 7, 7, 512, (3, 3), 1, (1, 1), False),
    (32, 2048, 7, 7, 512, (1, 1), 1, (0, 0), False),
    (4, 3, 224, 224, 64, (7, 7), 2, (3, 3), False),
    (2, 96, 17, 13, 72, (3, 3), 1, (1, 1), True),     # ragged everything, Cout not a tile multiple
    (1, 32, 5, 5, 8, (5, 5), 1, (2, 2), True),
    (2, 40, 9, 9, 24, (3, 3), 1, (0, 0), False),      # Cin % 32 != 0 -> flat form
    (2, 64, 12, 12, 130, (1, 1), 1, (0, 0), True),
    # non-square kernels in the channel-block form: the loader's (kh, kw) cursor against the producer's tap index
    (2, 32, 9, 11, 40, (1, 3), 1, (0, 1), True),      # 3 boxes: odd chain count
    (2, 32, 11, 9, 96, (3, 1), 1, (1, 0), False),     # 3 boxes, Cout 96 without bias
    (1, 64, 13, 13, 65, (1, 7), 1, (0, 3), True),     # Cout 65: TN 128 with one channel in its second half
    (1, 64, 13, 12, 100, (7, 1), 2, (3, 0), True),
    (2, 64, 10, 12, 129, (5, 3), 1, (2, 1), False),   # Cout 129: a second channel tile of one channel
    # padding larger than k // 2: output rows / columns made of padding and bias only
    (2, 64, 6, 7, 64, (3, 3), 1, (2, 3), True),       # Cout 64 with bias: a full TN 64 tile through the ragged store
    (1, 16, 5, 5, 8, (3, 3), 1, (3, 3), False),       # flat; the padding-only outputs must be exact zeros
    # stride >= 3, stride larger than the kernel, (H + 2p - K) % stride != 0
    (2, 64, 17, 17, 1, (2, 2), 4, (0, 0), True),      # Cout 1
    (3, 32, 20, 19, 33, (1, 1), 3, (0, 0), False),    # one box: a chain shorter than two boxes
    (2, 3, 23, 22, 8, (2, 2), 3, (1, 0), True),       # flat_rows<1> (KW 2)
    (2, 40, 9, 10, 24, (3, 3), 2, (1, 0), False),     # flat_rows<2>; input column 9 is outside every window
    # the other flat-form row widths and the flat-K limit
    (1, 3, 19, 27, 16, (3, 9), 4, (1, 0), True),      # flat_rows<4> (KW 9 of 16), columns 25-26 outside every window
    (1, 2, 10, 30, 5, (1, 16), 1, (0, 8), False),     # flat_rows<4>, a full 16-tap row
    (2, 12, 11, 13, 20, (3, 5), 2, (0, 2), False),    # flat_rows<3> (KW 5 of 8)
    (2, 16, 12, 15, 72, (4, 8), 1, (2, 3), True),     # Cin*KH*KWP == 512: the kernel-row table full, 16 boxes
    (2, 24, 9, 10, 48, (5, 3), 1, (2, 1), True),      # flat, non-square
    # box counts of the channel-block form
    (2, 32, 7, 9, 64, (1, 1), 1, (0, 0), False),      # one box; Cout 64 without bias: the unguarded store
    (2, 96, 9, 7, 128, (1, 1), 1, (0, 0), True),      # 3 boxes, a full TN 128 tile with bias
    (1, 64, 9, 9, 65, (7, 7), 1, (3, 3), False),      # 49 taps in the weight tensor map, Cout 65 without bias
    # output-channel tiles
    (2, 40, 6, 6, 1, (1, 1), 1, (0, 0), False),       # flat_rows<0>, Cout 1 without bias
    (2, 64, 8, 8, 96, (3, 3), 1, (1, 1), True),
    (2, 64, 8, 8, 100, (1, 1), 1, (0, 0), False),
    (1, 32, 9, 9, 129, (3, 3), 2, (1, 1), True),
    # fewer than 128 output positions: one partial M tile
    (1, 64, 5, 5, 96, (3, 3), 3, (1, 1), True),
    # more work items than SMs (50 position tiles x 2 channel tiles x 2 models): persistent CTAs walk both problems
    (4, 64, 40, 40, 129, (1, 3), 1, (0, 1), True),
]


def _case_id(c):
    """Square kernels and symmetric padding print as one number, as the cases of the ResNet family always have."""
    nb, cin, h, w, cout, (kh, kw), stride, (ph, pw), bias = c
    k = kh if kh == kw else (kh, kw)
    p = ph if ph == pw else (ph, pw)
    return str((nb, cin, h, w, cout, k, stride, p, bias))


def _mods(cin, cout, k, stride, pad, bias, seed):
    torch.manual_seed(seed)
    m = torch.nn.Conv2d(cin, cout, k, stride, pad, bias=bias).cuda()
    return m


def _ref(x, m):
    """fp64 convolution of module ``m`` on ``x`` and the condition bound B = conv(|x|, |w|) + |bias| of each output."""
    w, b = m.weight.double(), None if m.bias is None else m.bias.double()
    xd = x.double()
    y64 = F.conv2d(xd, w, b, m.stride, m.padding)
    bound = F.conv2d(xd.abs(), w.abs(), None if b is None else b.abs(), m.stride, m.padding)
    return y64, bound


def _errors(y, ref, bound, slack=None):
    """(max over outputs of (|y - ref| - slack) / bound, max|y - ref| / max|ref|); an output with a zero bound
    must match exactly (inf otherwise), so must every output that is not finite."""
    d = (y.double() - ref).abs()
    if slack is not None:
        d = (d - slack).clamp_min(0.0)
    d = torch.where(torch.isfinite(y), d, torch.full_like(d, float("inf")))
    ratio = torch.where(bound > 0, d / bound.clamp_min(1e-300), torch.where(d > 0, float("inf"), 0.0))
    return ratio.max().item(), (y.double() - ref).abs().max().item() / ref.abs().max().item()


def _check(y, ref, bound, slack=None, global_tol=GLOBAL_TOL, global_floor=0.0):
    """The kernel's output against its fp64 reference: |y - ref| <= TOL * bound + slack for every output, and
    max|y - ref| <= global_tol * max(max|ref|, global_floor)."""
    assert y.shape == ref.shape
    ratio, glob = _errors(y, ref, bound, slack)
    assert ratio <= TOL, f"elementwise: max |y - y64| / B = {ratio:.3g} > {TOL:g}"
    scale = max(1.0, global_floor / ref.abs().max().item())
    assert glob <= global_tol * scale, f"global: max |y - y64| / max |y64| = {glob:.3g}"


def _unread_mask(h, w, kh, kw, stride, ph, pw):
    """[h, w] bool: input positions outside every window of the convolution (a ragged tail, the gaps of a stride
    larger than the kernel)."""
    def covered(n, k, p):
        c = torch.zeros(n, dtype=torch.bool)
        for o in range((n + 2 * p - k) // stride + 1):
            lo = o * stride - p
            c[max(lo, 0):max(min(lo + k, n), 0)] = True
        return c

    return ~(covered(h, kh, ph)[:, None] & covered(w, kw, pw)[None, :])


@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_conv_pair_matches_fp64(case):
    """Both models in one launch (different weights and inputs), then the single-problem launch.  Input b has a
    large mean, so the outputs cancel; input a holds +inf wherever no window reads it (a kernel that reads past its
    windows, e.g. over the zero-weight taps of a flat-form row, turns it into NaN)."""
    from pleas_merging_b200 import conv

    nb, cin, h, w, cout, k, stride, pad, bias = case
    ma, mb = _mods(cin, cout, k, stride, pad, bias, 1), _mods(cin, cout, k, stride, pad, bias, 2)
    g = torch.Generator(device="cuda").manual_seed(3)
    xa = torch.randn(nb, cin, h, w, device="cuda", generator=g)
    xb = torch.relu(torch.randn(nb, cin, h, w, device="cuda", generator=g)) * 3.0 + 5.0
    unread = _unread_mask(h, w, *k, stride, *pad).cuda()
    xa_inf = xa.masked_fill(unread, float("inf"))
    assert conv.eligible(ma)
    pair = conv.ConvPair(ma, mb)
    with torch.no_grad():
        ya, yb = pair(xa_inf, xb)
        for y, m, x in ((ya, ma, xa), (yb, mb, xb)):
            _check(y, *_ref(x, m))
        # single-problem launch
        y1 = conv.conv2d(xa_inf, ma)
        assert torch.equal(y1, ya)


def test_conv_weight_update_is_seen():
    from pleas_merging_b200 import conv

    m = _mods(64, 64, 3, 1, 1, False, 0)
    x = torch.randn(2, 64, 8, 8, device="cuda")
    pk = conv.PackedConv(m)
    with torch.no_grad():
        y0 = conv.conv2d(x, m, pk)
        m.weight.mul_(2.0)
        y1 = conv.conv2d(x, m, pk)
    assert torch.allclose(y1, 2 * y0, rtol=1e-5, atol=1e-6)


def test_conv_ineligible_falls_back_to_module():
    from pleas_merging_b200 import conv

    m = torch.nn.Conv2d(64, 64, 3, 1, 1, groups=2).cuda()
    assert not conv.eligible(m)
    x = torch.randn(1, 64, 8, 8, device="cuda")
    with torch.no_grad():
        assert torch.equal(conv.conv2d(x, m), m(x))


@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("case", [(2, 64, 28, 28, 256, (1, 1), 1, (0, 0), False),
                                  (3, 64, 14, 14, 72, (3, 3), 1, (1, 1), True),
                                  (2, 3, 32, 32, 24, (7, 7), 2, (3, 3), False),
                                  (2, 64, 10, 11, 48, (5, 3), 1, (1, 2), False),
                                  (2, 64, 9, 9, 100, (3, 3), 1, (1, 1), True)],
                         ids=["1x1", "3x3-ragged", "stem", "5x3-asym-pad", "cout100-bias"])
def test_conv_with_fused_batchnorm_relu_output(case, relu):
    """plb_conv2d_affine_forward: the eval-mode BatchNorm (+ ReLU) behind a convolution as a second output of the same
    launch, against the fp64 modules; the first output stays the plain convolution.  The second output
    z = relu?(s y + t) is held to TOL * |s| B plus 2^-24 |t|, the fp32 rounding of the shift."""
    from pleas_merging_b200 import conv

    nb, cin, h, w, cout, k, stride, pad, bias = case
    mods, bns = [], []
    for seed in (1, 2):
        torch.manual_seed(seed)
        mods.append(torch.nn.Conv2d(cin, cout, k, stride, pad, bias=bias).cuda())
        bn = torch.nn.BatchNorm2d(cout).cuda().eval()
        with torch.no_grad():
            bn.weight.copy_(torch.randn(cout).cuda())        # negative scales included
            bn.bias.copy_(0.3 * torch.randn(cout).cuda())
            bn.running_mean.copy_(0.2 * torch.randn(cout).cuda())
            bn.running_var.copy_(0.5 + torch.rand(cout).cuda())
        bns.append(bn)
    xa, xb = torch.randn(nb, cin, h, w, device="cuda"), torch.randn(nb, cin, h, w, device="cuda")
    pair = conv.ConvPair(mods[0], mods[1], bns=tuple(bns), relu=relu)
    with torch.no_grad():
        ya, yb, za, zb = pair(xa, xb)
        for y, z, m, bn, x in ((ya, za, mods[0], bns[0], xa), (yb, zb, mods[1], bns[1], xb)):
            ref, bound = _ref(x, m)
            ref2 = F.batch_norm(ref, bn.running_mean.double(), bn.running_var.double(), bn.weight.double(),
                                bn.bias.double(), False, 0.0, bn.eps)
            if relu:
                ref2 = torch.relu(ref2)
            s = bn.weight.double() * (bn.running_var.double() + bn.eps).rsqrt()
            t = bn.bias.double() - bn.running_mean.double() * s
            _check(y, ref, bound)
            _check(z, ref2, s.abs().view(-1, 1, 1) * bound, slack=2.0 ** -24 * t.abs().view(-1, 1, 1),
                   global_tol=4e-6, global_floor=1.0)
        # a BatchNorm update is seen by the next call
        bns[0].running_mean.add_(1.0)
        _, _, za2, _ = pair(xa, xb)
        assert not torch.equal(za2, za)


GRID_K = (1, 2, 3, 5, 8, 9, 16, 17)
GATE_POINTS = {f"cin{cin}": [(cin, kh, kw) for kh in GRID_K for kw in GRID_K] for cin in (3, 16, 31, 32, 40, 64)}
# either side of the flat form's K = Cin * KH * pow2(KW) <= 512: 512, 544, 1024, 480, 528, 512 (496 padded to a box)
GATE_POINTS["flat-k-limit"] = [(16, 4, 8), (17, 4, 8), (16, 4, 9), (3, 10, 16), (3, 11, 16), (31, 1, 16)]


@pytest.mark.parametrize("stride", [1, 2, 3])
@pytest.mark.parametrize("points", list(GATE_POINTS.values()), ids=list(GATE_POINTS))
def test_conv_gate_and_kernel_agree(points, stride):
    """What ``conv.eligible()`` admits runs on the kernel (one launch) and meets both bars; everything else is the
    module's own forward, bit for bit, with no launch."""
    from pleas_merging_b200 import _native as N
    from pleas_merging_b200 import conv

    g = torch.Generator(device="cuda").manual_seed(5)
    admitted = 0
    for cin, kh, kw in points:
        m = _mods(cin, 8, (kh, kw), stride, (kh // 2, kw // 3), True, kh * 100 + kw)
        x = torch.randn(2, cin, kh + 5, kw + 6, device="cuda", generator=g)
        before = N.LAUNCH_COUNTS["plb_conv2d_affine_forward"]
        with torch.no_grad():
            y = conv.conv2d(x, m)
            launches = N.LAUNCH_COUNTS["plb_conv2d_affine_forward"] - before
            if conv.eligible(m):
                admitted += 1
                assert launches == 1, (cin, kh, kw)
                _check(y, *_ref(x, m))
            else:
                assert launches == 0, (cin, kh, kw)
                assert torch.equal(y, m(x)), (cin, kh, kw)
    assert admitted > 0


@pytest.mark.parametrize("points", list(GATE_POINTS.values()), ids=list(GATE_POINTS))
def test_conv_gate_matches_c_abi(points):
    """``conv.eligible()`` (MAX_FLAT_K, its pow2(KW) formula) agrees with conv_geometry() and the checks of the C ABI:
    plb_conv_pack_weights packs exactly the admitted weights and refuses the others with PLB_ESIZE."""
    from pleas_merging_b200 import _native as N
    from pleas_merging_b200 import conv

    lib = N.lib()
    stream = torch.cuda.current_stream().cuda_stream
    for cin, kh, kw in points:
        m = torch.nn.Conv2d(cin, 1, (kh, kw), bias=False).cuda()
        packed = torch.empty(lib.plb_conv_packed_floats(1, cin, kh, kw), device="cuda")
        rc = lib.plb_conv_pack_weights(m.weight.data_ptr(), 1, cin, kh, kw, packed.data_ptr(), stream)
        assert rc in (0, PLB_ESIZE), (cin, kh, kw, rc)
        assert (rc == 0) == conv.eligible(m), (cin, kh, kw, rc)
    torch.cuda.synchronize()


def test_conv_input_over_2_31_elements():
    """One convolution over an input (and, for the 1x1, an output) of more than 2^31 elements: per-image offsets
    must be 64-bit.  Images are independent, so the first, the last and the one that straddles element 2^31 are
    checked on their own against fp64."""
    from pleas_merging_b200 import _native as N
    from pleas_merging_b200 import conv

    nb, cin, h, w = 700, 64, 224, 224
    assert nb * cin * h * w > 2 ** 31
    straddle = 2 ** 31 // (cin * h * w)
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(nb, cin, h, w, device="cuda", generator=g)
    for k, stride, pad in ((1, 1, 0), (3, 2, 1)):
        m = _mods(cin, 64, k, stride, pad, True, k)
        before = N.LAUNCH_COUNTS["plb_conv2d_affine_forward"]
        with torch.no_grad():
            y = conv.conv2d(x, m)
        assert N.LAUNCH_COUNTS["plb_conv2d_affine_forward"] == before + 1
        for n in (0, straddle, nb - 1):
            _check(y[n:n + 1], *_ref(x[n:n + 1], m))
        del y
    del x
    torch.cuda.empty_cache()
