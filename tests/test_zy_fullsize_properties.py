"""GPU: parity at BASELINE.json's FULL size (LLaMA-7B shapes, 131072 tokens, 1 % outliers) through size-independent
properties -- the oracle cannot finish a 128K-token layer in seconds, so the full-size checks are
  * the fused attend == the legacy two-op chain (K op -> softmax -> V op), whose ops are oracle-checked at small sizes;
  * the device-resident-length attend == the host-length attend;
  * linearity of the K op in q and of the V op in the scores;
  * our legacy ops == the reference's own CUDA kernels on the same seeded cache (their results are stored in
    tests/golden/refgpu_fullsize.npz by tests/golden/gen_refgpu_golden.py: the V outputs whole, the K scores as a
    fixed sample of 16384 elements plus per-head sums and norms over all of them).
Tolerance 1e-4 relative to the result's scale (fp32 accumulation order; the probe measures 1e-7 .. 1e-6).
The file name keeps it after the small-size parity tests in the collection order."""
import numpy as np
import pytest
import torch

from _util import golden_rel_err, load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
L, H = 131072, 32
TOL = 1e-4


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def fill(bits):
    from kvquant_b200 import synth, cache as kc
    sp = synth.SynthSpec(H, 128, seed=0)
    cal = synth.calibrate(sp, bits, calib_tokens=512, seed=7)
    klut = kc.build_k_lookup_table(cal["k"][0], cal["k"][1], cal["k"][2][0], H, device=DEV)
    lc = kc.LayerCache.from_luts(bits, H, L + 64, dict(lut=klut["lut"], lut2=None, thr_lower=klut["thr_lower"],
                                                      thr_upper=klut["thr_upper"]), cal["v"][2][0], device=DEV)
    synth.fill_layer_cache_gpu(lc, sp, L, seed=bits)
    torch.cuda.synchronize()
    return lc


@pytest.fixture(scope="module", params=[4, 3])
def filled(request):
    bits = request.param
    lc = fill(bits)
    yield bits, lc
    del lc
    torch.cuda.empty_cache()


KNAME = "vecquant%dmatmul_nuq_perchannel_transposed_rope_mha_batched_fused_opt2"
VNAME = "vecquant%dmatmul_nuq_perchannel_transposed_mha_batched_fused_opt2"


def _ops(bits, mod=None):
    if mod is None:
        from kvquant_b200 import quant_cuda as mod
    return getattr(mod, KNAME % bits), getattr(mod, VNAME % bits)


def _k(lc, op, q):
    mul = torch.zeros((1, H, L), device=DEV)
    op(q, lc.kcache, mul, lc.klut.view(H, 128, -1), L, lc.k_outliers, lc.k_outlier_idx, 10000.0, 0)
    return mul


def _v(lc, op, p):
    mul = torch.zeros((1, H, 128), device=DEV)
    op(p, lc.vcache, mul, lc.vlut, L, lc.v_outliers, lc.v_outlier_idx)
    return mul


def test_fused_attend_equals_the_two_op_chain_and_the_device_length_form(filled):
    bits, lc = filled
    k2, v2 = _ops(bits)
    g = torch.Generator(device=DEV).manual_seed(1)
    q = torch.randn((1, H, 128), generator=g, device=DEV).half().float()
    s = _k(lc, k2, q)
    p = torch.softmax(s[0] / np.sqrt(128), -1)[None].contiguous()
    chain = _v(lc, v2, p)[0]
    len_dev = torch.full((1,), L - 1, dtype=torch.int64, device=DEV)
    # exact "ratio" tables (the default) / north_star's fp16 tables.  The fp16 mode does NOT meet 1e-3 at this length:
    # measured 1.4e-3 .. 2.2e-3 of the output scale (up to 9e-3 of a single head's own scale) -- the fp16 rounding of the
    # K table entries and of cos/sin moves every softmax weight by ~8e-4, and at 128K nothing averages that away
    # (the reference's own chain rounds the scores to fp16, which moves them by up to 3e-3).  Bounds = 1.5x measured.
    for precision, tol, tol_head in (("fp32", TOL, 3 * TOL), ("fp16", 3.5e-3, 1.5e-2)):
        lc.precision = precision
        fused = lc.attend(q[0].contiguous()).clone()
        assert _rel(fused, chain) < tol, (precision, _rel(fused, chain))
        # per head, relative to that head's own scale
        d = ((fused - chain).abs().amax(dim=1) / chain.abs().amax(dim=1)).max().item()
        assert d < tol_head, (precision, d)
        dyn = lc.attend_dyn(q[0].contiguous(), len_dev, 1).clone()
        assert _rel(dyn, fused) < 5e-5   # same kernels and token ranges; only the order of the outlier reductions differs
    lc.precision = "fp32"


def test_k_op_is_linear_in_q_and_v_op_in_the_scores(filled):
    bits, lc = filled
    k2, v2 = _ops(bits)
    g = torch.Generator(device=DEV).manual_seed(2)
    q1 = torch.randn((1, H, 128), generator=g, device=DEV)
    q2 = torch.randn((1, H, 128), generator=g, device=DEV)
    lhs = _k(lc, k2, (q1 + 0.5 * q2).contiguous())
    rhs = _k(lc, k2, q1) + 0.5 * _k(lc, k2, q2)
    assert _rel(lhs, rhs) < TOL
    p1 = torch.rand((1, H, L), generator=g, device=DEV)
    p2 = torch.rand((1, H, L), generator=g, device=DEV)
    lhs = _v(lc, v2, (2.0 * p1 + p2).contiguous())
    rhs = 2.0 * _v(lc, v2, p1) + _v(lc, v2, p2)
    assert _rel(lhs, rhs) < TOL


def legacy_ops(bits, lc, mod=None):
    """K op scores and V op output on seeded inputs."""
    k2, v2 = _ops(bits, mod)
    g = torch.Generator(device=DEV).manual_seed(3)
    q = torch.randn((1, H, 128), generator=g, device=DEV).half().float()
    p = torch.softmax(torch.randn((1, H, L), generator=g, device=DEV) * 2, -1).half().float()
    return {"k": _k(lc, k2, q), "v": _v(lc, v2, p)}


def test_legacy_ops_equal_the_reference_kernels_at_full_size(filled):
    bits, lc = filled
    g = load_golden("refgpu_fullsize.npz")
    for key, t in legacy_ops(bits, lc).items():
        e_norm, _, e_sums = golden_rel_err(g, "b%d" % bits, key, t)
        assert e_norm < TOL and e_sums < TOL, (key, e_norm, e_sums)
