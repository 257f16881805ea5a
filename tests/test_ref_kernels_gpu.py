"""GPU parity, kernel against kernel: the product's sm_100a kernels (through the C-ABI) versus what the reference's OWN CUDA ops
computed on a B200 for the same seeded inputs -- the UNMODIFIED sources under ops/ctc_2d/csrc and assets/ops/dcn/src, compiled by
oracle/build_ref.py and run by `python -m oracle.make_golden ref_kernels` into tests/golden/ref_kernels.npz (SURVEY.md section
8c's "third check").  This is the pin for every native op of the path: 2D-CTC K1/K2/K3 in fp32 and fp64 incl. the realistic
(saturating-python) cfg-3 regime, DCNv1/v2 incl. the offset-size != output-size quirk, and deformable PS-RoI pooling (row A13).
The same inputs also go through the CPU restatements in oracle/*.c, so the oracle itself is pinned to the reference here.

The reference outputs reach 136 MB per case, so the golden file keeps, for each array, CRC-32 hashes of its whole -inf and zero
masks, its finite / zero counts, largest magnitude and L2 norm, and a fixed seeded sample of its values.  Where more than half of
an array is zero or -inf (CTC gradients and log_alpha, the DCN gradients of out-of-range samples) the sample is drawn from its
finite nonzero entries, all of them when they are few (at most 8192 and at most 1/16 of the array), so that scattered values
are compared one by one; the positions follow from the masks, which are checked first.  Otherwise the sample is uniform.  The
whole-array statistics are compared within the bounds that the elementwise tolerance implies for every entry.  The deformable
pooling outputs are small and kept whole.  The "provenance" entry names the GPU, driver, torch and reference binaries of the
recording."""
import os
import zlib

import numpy as np
import pytest
import torch

from oracle import capi
from tests.cases import ctc2d_case
from tests.deform_pool_cases import CASES as POOL_CASES, make as pool_make

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "ref_kernels.npz")
SAMPLE = 256              # sampled entries of each large reference output kept in the golden file
WHOLE = 8192              # a sparse array's nonzero entries are kept whole up to this many


@pytest.fixture(scope="module")
def gold():
    with np.load(GOLD) as g:
        return dict(g)


def _dev(cuda, *arrs):
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda) for a in arrs]


def _choice(size, key):
    rng = np.random.RandomState(zlib.crc32(key.encode()))
    return np.sort(rng.choice(size, min(size, SAMPLE), replace=False))


def _masks(flat):
    fin, zero = np.isfinite(flat), flat == 0
    return fin, zero, [float(zlib.crc32(np.packbits(m).tobytes())) for m in (fin, zero)]


def _sample_index(flat, key, nonzero_mode):
    if not nonzero_mode:
        return _choice(flat.size, key)
    nz = np.flatnonzero(np.isfinite(flat) & (flat != 0))
    if nz.size <= WHOLE and 16 * nz.size <= flat.size:
        return nz
    return nz[_choice(nz.size, key)]


def record(out, key, a):
    """Golden entries of one reference output (oracle/make_golden.py): the sample, and [finite count, zero count, max |.|, L2 norm,
    CRC-32 of the finite mask, CRC-32 of the zero mask, 1 if the sample is drawn from the finite nonzero entries]."""
    flat = np.asarray(a).reshape(-1)
    fin, zero, crcs = _masks(flat)
    vals = flat[fin].astype(np.float64)
    nonzero_mode = 2 * int((fin & ~zero).sum()) < flat.size
    out[key] = flat[_sample_index(flat, key, nonzero_mode)]
    out[key + ".stats"] = np.array([vals.size, zero.sum(), np.abs(vals).max() if vals.size else 0.0, np.linalg.norm(vals)] + crcs
                                   + [float(nonzero_mode)])


def check(a, gold, key, rtol, atol, patterns=False, like=None, what=""):
    """`a` against the reference output recorded under `key`, as assert_allclose(a, ref, rtol, atol) would see it: the sample
    entry by entry, and over the whole array |max|a| - max|ref|| <= atol + rtol max|ref| and
    | ||a|| - ||ref|| | <= atol sqrt(n) + rtol ||ref||.  patterns=True requires the same -inf and zero masks (counts and hashes).
    like: an array already checked with patterns=True against the same reference output; its masks then stand for the
    reference's, and `a` must stay within atol of zero wherever the reference is zero."""
    flat = np.asarray(a).reshape(-1)
    n_finite, n_zeros, mx, l2, crc_fin, crc_zero, nonzero_mode = gold[key + ".stats"]
    fin, zero, crcs = _masks(flat)
    if patterns:
        assert fin.sum() == n_finite, "%s: -inf count differs from the reference kernel" % what
        assert zero.sum() == n_zeros, "%s: zero count differs from the reference kernel" % what
        assert crcs[0] == crc_fin, "%s: -inf positions differ from the reference kernel" % what
        assert crcs[1] == crc_zero, "%s: zero positions differ from the reference kernel" % what
    ref_flat = flat if like is None else np.asarray(like).reshape(-1)
    if like is not None:
        assert _masks(ref_flat)[2] == [crc_fin, crc_zero], "%s: `like` does not carry the reference's masks" % what
        ref_zero = ref_flat == 0
        assert np.all(np.abs(flat[ref_zero]) <= atol), "%s: nonzero where the reference kernel is zero" % what
    elif nonzero_mode:
        assert patterns, "%s: a nonzero-entry sample needs the reference's masks (patterns=True or like=)" % what
    got, ref = flat[_sample_index(ref_flat, key, bool(nonzero_mode))], gold[key]
    assert got.shape == ref.shape, what
    sel = np.isfinite(ref)
    np.testing.assert_allclose(got[sel], ref[sel], rtol=rtol, atol=atol, err_msg=what)
    vals = flat[fin].astype(np.float64)
    assert abs(float(np.abs(vals).max() if vals.size else 0.0) - mx) <= atol + rtol * mx, "%s: max |.|" % what
    assert abs(float(np.linalg.norm(vals)) - l2) <= atol * np.sqrt(vals.size) + rtol * l2, "%s: L2 norm" % what


# ------------------------------------------------------------------------------------------------ 2D-CTC
CTC_CASES = [
    # seed, T, H, N, C, S, Lmax, ragged, peak
    (31, 32, 8, 64, 38, 32, 12, False, 0.0),    # cfg-3 shape, random logits: loss ~ 90-130 (python reference saturates here)
    (32, 32, 8, 33, 38, 32, 16, True, 0.0),     # ragged input lengths, longest targets
    (33, 32, 8, 16, 38, 32, 12, False, 6.0),    # peaked (trained-model-like) regime
    (34, 16, 4, 9, 11, 8, 6, True, 0.0),
    (35, 64, 1, 5, 38, 32, 20, False, 0.0),     # H = 1 (1D CTC through the 2D op)
    (36, 8, 3, 3, 4001, 4, 4, False, 0.0),      # large alphabet
    (37, 32, 8, 2048, 38, 32, 12, False, 0.0),  # the CRNN-2D head's batch
    (38, 32, 8, 6, 5000, 32, 32, True, 0.0),    # ChineseCharset-sized alphabet at the real T / H, targets up to 32 labels
    (39, 32, 8, 11, 38, 32, 32, False, 0.0),    # longest targets (65 states: 3 states per lane, slot rounds)
]
CTC_DTYPES = {"f32": np.float32, "f64": np.float64}


def ctc_skip_reason(case, dtype):
    N, C = case[3], case[4]
    if dtype == np.float64 and N > 256:
        return "fp64 at the large batch adds nothing"
    if dtype == np.float64 and C > 1024:
        return "fp64 with a >1k-class alphabet: the fp64 DP keeps [T, C] rows on chip -> MR_ERR_UNSUPPORTED (DESIGN.md section 7)"
    return None


def ctc_inputs(case, dtype):
    seed, T, H, N, C, S, Lmax, ragged, peak = case
    assert 1024 % T == 0
    lp, tg, il, tl = ctc2d_case(seed, T, H, N, C, S, Lmax, peak=peak, ragged_T=ragged, dtype=dtype)
    return lp, tg, il, tl, (1.0 / tl).astype(dtype)


@pytest.mark.parametrize("dtype", list(CTC_DTYPES.values()), ids=list(CTC_DTYPES))
@pytest.mark.parametrize("case", CTC_CASES, ids=[str(c[0]) for c in CTC_CASES])
def test_ctc2d_vs_reference_kernels(cuda, gold, case, dtype):
    """ops/ctc_2d/csrc/cuda/ctc2d_cuda_kernel.cu K1 (:54-211), K2 (:254-368), K3 (:427-517) as they ran on a B200.  T divides 1024
    in every case, so the reference's K3 aliasing race (SURVEY App. B1.5) is not in play and its output is deterministic."""
    from megreader_b200 import ctc2d
    if ctc_skip_reason(case, dtype):
        pytest.skip(ctc_skip_reason(case, dtype))
    N, C = case[3], case[4]
    key = "ctc.%d.%s" % (case[0], "f32" if dtype == np.float32 else "f64")
    lp, tg, il, tl, go = ctc_inputs(case, dtype)
    d_lp, d_tg, d_il, d_tl, d_go = _dev(cuda, lp, tg, il, tl, go)
    nll, la = ctc2d.ctc2d_forward(d_lp, d_tg, d_il, d_tl, 0, 0.0)
    gr = ctc2d.ctc2d_backward(d_go, d_lp, d_tg, d_il, d_tl, nll, la, 0)
    rt = 1e-4 if dtype == np.float32 else 1e-9
    grt, gat = (2e-4, 2e-5) if dtype == np.float32 else (1e-8, 1e-10)
    r_nll = gold[key + ".nll"]
    nll, la, gr = [t.cpu().numpy() for t in (nll, la, gr)]
    assert np.isfinite(r_nll).all()
    np.testing.assert_allclose(nll, r_nll, rtol=rt)
    check(la, gold, key + ".log_alpha", rt, 1e-4 if dtype == np.float32 else 1e-9, patterns=True, what="log_alpha")
    check(gr, gold, key + ".grad", grt, gat, patterns=True, what="grad")
    # training pair (what ops.ctc_loss_2d runs when log_probs requires grad): same values
    if dtype == np.float32:
        x = d_lp.clone().requires_grad_(True)
        loss = ctc2d.ctc_loss_2d(x, d_tg, d_il, d_tl)
        (loss * d_go).sum().backward()
        np.testing.assert_allclose(loss.detach().cpu().numpy(), r_nll, rtol=rt)
        check(x.grad.cpu().numpy(), gold, key + ".grad", 2e-4, 2e-5, like=gr, what="training-pair grad")
    # and the CPU restatement is pinned to the same reference output (small cases: the C oracle is serial)
    if N <= 64 and C <= 64:
        o_nll, o_la = capi.ctc2d_forward(lp.astype(np.float64), tg, il, tl)
        o_gr = capi.ctc2d_backward(go.astype(np.float64), lp.astype(np.float64), tg, il, tl, o_nll, o_la)
        np.testing.assert_allclose(o_nll, r_nll, rtol=rt)
        check(o_gr, gold, key + ".grad", grt, gat, like=gr, what="oracle grad")


# ------------------------------------------------------------------------------------------------ DCN v1 / v2
def _dcn_inputs(seed, B, C, H, W, Cout, k, s, p, d, group, dg, big_offset):
    rng = np.random.RandomState(seed)
    Ho = (H + 2 * p - (d * (k - 1) + 1)) // s + 1
    Wo = (W + 2 * p - (d * (k - 1) + 1)) // s + 1
    oh, ow = (H, W) if big_offset else (Ho, Wo)
    x = rng.standard_normal((B, C, H, W)).astype(np.float32)
    w = (rng.standard_normal((Cout, C // group, k, k)) / np.sqrt(C * k * k)).astype(np.float32)
    b = rng.standard_normal((Cout,)).astype(np.float32)
    off = (rng.standard_normal((B, 2 * k * k * dg, oh, ow)) * 1.5).astype(np.float32)
    m = (1 / (1 + np.exp(-rng.standard_normal((B, k * k * dg, oh, ow))))).astype(np.float32)
    go = rng.standard_normal((B, Cout, Ho, Wo)).astype(np.float32)
    return x, w, b, off, m, go, Ho, Wo


DCN_CASES = [
    # B, C, H, W, Cout, k, s, p, d, group, dg, with_bias, big_offset
    (2, 8, 9, 11, 8, 3, 1, 1, 1, 1, 1, True, False),
    (3, 8, 8, 8, 8, 3, 2, 1, 1, 1, 1, False, True),       # stride 2 with INPUT-sized offset/mask maps (SURVEY App. B2.1)
    (2, 16, 10, 7, 8, 3, 1, 2, 2, 2, 2, True, False),     # dilation 2, groups, deformable groups
    (4, 128, 16, 16, 128, 3, 1, 1, 1, 1, 1, False, False),
    (2, 256, 16, 16, 256, 3, 2, 1, 1, 1, 1, False, True),  # layer-3 first block geometry (stride 2, big offset)
    (2, 64, 12, 20, 64, 3, 1, 1, 1, 1, 1, True, False),
    (2, 128, 13, 19, 256, 3, 1, 1, 1, 1, 1, True, False),  # fused backward, ragged 8 x 16 tiles, Cout = 2 x 128
]
DCNV1_CASES = {"a": (4, 8, 9, 11, 8, 3, 1, 1, 1, 1, 1), "b": (4, 16, 12, 12, 8, 3, 2, 1, 1, 2, 2),
               "c": (2, 64, 16, 16, 64, 3, 1, 1, 1, 1, 1)}


def _close(a, gold, key, what, tol=1e-4):
    scale = max(1.0, float(gold[key + ".stats"][2]))
    check(a.cpu().numpy(), gold, key, tol, tol * scale, patterns=bool(gold[key + ".stats"][6]), what=what)


@pytest.mark.parametrize("case", DCN_CASES, ids=[str(i) for i in range(len(DCN_CASES))])
def test_dcnv2_vs_reference_kernels(cuda, gold, case):
    """assets/ops/dcn/src/deform_conv_cuda.cpp:486-679 + deform_conv_cuda_kernel.cu:569-766 as they ran on a B200."""
    from megreader_b200 import dcn
    key = "dcn2.%d." % DCN_CASES.index(case)
    B, C, H, W, Cout, k, s, p, d, group, dg, with_bias, big = case
    x, w, b, off, m, go, Ho, Wo = _dcn_inputs(11, B, C, H, W, Cout, k, s, p, d, group, dg, big)
    tx, tw, tb, toff, tm, tgo = _dev(cuda, x, w, b, off, m, go)
    out = tx.new_empty(B, Cout, Ho, Wo)
    dcn.modulated_deform_conv_cuda_forward(tx, tw, tb, None, toff, tm, out, None, k, k, s, s, p, p, d, d, group, dg, with_bias)
    gi, gw, gb, goff, gm = [torch.zeros_like(t) for t in (tx, tw, tb, toff, tm)]
    dcn.modulated_deform_conv_cuda_backward(tx, tw, tb, None, toff, tm, None, gi, gw, gb, goff, gm, tgo, k, k, s, s, p, p, d, d,
                                            group, dg, with_bias)
    _close(out, gold, key + "output", "output")
    _close(gi, gold, key + "grad_input", "grad_input")
    _close(gw, gold, key + "grad_weight", "grad_weight")
    _close(goff, gold, key + "grad_offset", "grad_offset")
    _close(gm, gold, key + "grad_mask", "grad_mask")
    if with_bias:
        _close(gb, gold, key + "grad_bias", "grad_bias")
    if big:   # the tail of each [., Hi, Wi] slab stays zero in both (flat (Ho,Wo) indexing)
        assert float(goff.view(B, -1)[:, 2 * k * k * dg * Ho * Wo:].abs().max()) == 0.0
        assert float(gold[key + "grad_offset_tail_max_abs"]) == 0.0


@pytest.mark.parametrize("name", sorted(DCNV1_CASES))
def test_dcnv1_vs_reference_kernels(cuda, gold, name):
    """deform_conv_{forward,backward_input,backward_parameters}_cuda, deform_conv_cuda.cpp:151-484 (K5-K7)."""
    from megreader_b200 import dcn
    key = "dcn1.%s." % name
    B, C, H, W, Cout, k, s, p, d, group, dg = DCNV1_CASES[name]
    x, w, _, off, _, go, Ho, Wo = _dcn_inputs(12, B, C, H, W, Cout, k, s, p, d, group, dg, False)
    tx, tw, toff, tgo = _dev(cuda, x, w, off, go)
    txg, toffg, twg = [t.clone().requires_grad_(True) for t in (tx, toff, tw)]
    out = dcn.deform_conv(txg, toffg, twg, s, p, d, group, dg)
    out.backward(tgo)
    _close(out.detach(), gold, key + "output", "output")
    _close(txg.grad, gold, key + "grad_input", "grad_input")
    _close(toffg.grad, gold, key + "grad_offset", "grad_offset")
    _close(twg.grad, gold, key + "grad_weight", "grad_weight")


# ------------------------------------------------------------------------------------------------ deformable PS-RoI pooling
def pool_args(a):
    return (int(a["no_trans"]), float(a["spatial_scale"]), a["output_dim"], a["group_size"], a["pooled"], a["part_size"],
            a["sample_per_part"], float(a["trans_std"]))


def pool_grad_out(n, od, P):
    return np.random.RandomState(1).standard_normal((n, od, P, P)).astype(np.float32)


@pytest.mark.parametrize("name", sorted(POOL_CASES))
def test_deform_pool_vs_reference_kernels(cuda, gold, name):
    """assets/ops/dcn/src/deform_pool_cuda_kernel.cu:52-263 (K11/K12) as they ran on a B200: pins row A13 and, through the same
    inputs, oracle/deform_pool_oracle.c."""
    from megreader_b200 import deform_pool as dp
    key = "pool.%s." % name
    data, rois, trans, a = pool_make(name)
    d, r = _dev(cuda, data.astype(np.float32), rois.astype(np.float32))
    t = _dev(cuda, trans.astype(np.float32))[0] if trans is not None else d.new_empty(0)
    n, od, P = rois.shape[0], a["output_dim"], a["pooled"]
    go = torch.from_numpy(pool_grad_out(n, od, P)).to(cuda)
    r_out, r_cnt, r_gin, r_gtr = [torch.from_numpy(gold[key + k]).to(cuda) for k in ("out", "count", "grad_input", "grad_trans")]
    out, cnt = d.new_zeros(n, od, P, P), d.new_zeros(n, od, P, P)
    dp.deform_psroi_pooling_cuda_forward(d, r, t, out, cnt, *pool_args(a))
    gin, gtr = torch.zeros_like(d), torch.zeros_like(t)
    dp.deform_psroi_pooling_cuda_backward(go, d, r, t, cnt, gin, gtr, *pool_args(a))
    # same fp32 arithmetic on both sides: the sample counts must agree exactly, values to rounding
    assert torch.equal(cnt, r_cnt), "top_count differs from the reference kernel"
    for got, ref, what, tol in ((out, r_out, "out", 1e-5), (gin, r_gin, "input_grad (atomic order differs)", 1e-4),
                                (gtr, r_gtr, "trans_grad", 1e-4)):
        if what == "trans_grad" and trans is None:
            continue
        got, ref = got.cpu().numpy(), ref.cpu().numpy()
        scale = max(1.0, float(np.abs(ref).max()))
        np.testing.assert_allclose(got, ref, rtol=tol, atol=tol * scale, err_msg=what)
    # the fp64 CPU restatement against the reference kernel (bins whose samples sit on a half-pixel border within fp32
    # rounding may count differently in fp64: they must be rare, and everything else must agree)
    o_out, o_cnt = capi.deform_psroi_forward(data, rois, trans, **a)
    same = o_cnt == gold[key + "count"]
    assert same.mean() > 0.98
    np.testing.assert_allclose(o_out[same], gold[key + "out"][same], rtol=1e-4, atol=1e-4)
