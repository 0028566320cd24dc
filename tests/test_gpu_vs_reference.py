"""GPU: our ops against the REFERENCE's own CUDA extension on the same inputs.

The reference results are stored in tests/golden/refgpu_vs_reference.npz: tests/golden/gen_refgpu_golden.py runs the
functions below with `mod` = the unmodified reference extension (deployment/kvquant/quant_cuda.cpp +
quant_cuda_kernel.cu compiled for sm_100a by oracle/build_ref.py); the tests run them with `mod` = this repository's
`quant_cuda` and compare.

Bars: packed codes / returned index arrays bit-exact; fp32 element-wise outputs bit-exact; matvecs within 2e-5
norm-wise (both sides accumulate in fp32, in different orders; the reference's own order is non-deterministic).
Reference defects are avoided, not reproduced: the 3-bit V prefill packer (quant_cuda_kernel.cu:2574-2579) and the
racy K prefill packer (1857-1883) are compared through the single-token ops instead.
"""
import numpy as np
import pytest
import torch

from _util import O, assert_bit_exact, golden_rel_err, load_golden, quantizer, spec

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN_FILE = "refgpu_vs_reference.npz"


@pytest.fixture(scope="module")
def g():
    return load_golden(GOLDEN_FILE)


@pytest.fixture(scope="module")
def qc():
    import quant_cuda
    return quant_cuda


def cu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def single_token_appends(mod, bits):
    klut, vcent = quantizer(bits)
    sp = spec()
    H, W, Lmax, T = 32, 128 * bits // 32, 64, 9
    k, v = sp.k_tokens(T, 41), sp.v_tokens(T, 42)
    lut = cu(klut["lut"].reshape(H, 128, -1))
    lo, hi = cu(klut["thr_lower"]), cu(klut["thr_upper"])
    kd, ks, vd, vs = [torch.zeros((H, W, Lmax), dtype=torch.int32, device=DEV) for _ in range(4)]
    vlut = torch.zeros((Lmax, 2 ** bits), dtype=torch.float32, device=DEV)
    rest = []
    for t in range(T):
        kv, vv = cu(k[t]), cu(v[t])
        getattr(mod, "vecquant%dappendvecK" % bits)(kd, lut, kv, t)
        r = kv.clone()
        getattr(mod, "vecquant%dappendvecKsparse" % bits)(ks, lut, kv, r, lo, hi, t)
        rest.append(r)
        thi, tlo, _, _ = O.v_thresholds(v[t], 21)
        lt = O.v_token_lut(vcent, thi, tlo)
        vlut[t] = cu(lt)
        getattr(mod, "vecquant%dappendvecV" % bits)(vd, vlut, vv, t)
        zp = float(lt[O.zero_point_code(bits)])
        getattr(mod, "vecquant%dappendvecVsparse" % bits)(vs, vlut, vv, zp, float(tlo), float(thi), t)
    return dict(kcache=kd, kcache_sparse=ks, k_residual=torch.stack(rest), vcache=vd, vcache_sparse=vs)


def prefill_v_packer(mod, bits):
    klut, vcent = quantizer(bits)
    sp = spec()
    H, W, Lmax, T = 32, 128 * bits // 32, 320, 300
    v = sp.v_tokens(T, 43)
    lo = np.zeros(T, np.float32); hi = np.zeros(T, np.float32)
    vlut = np.zeros((Lmax, 2 ** bits), np.float32)
    for t in range(T):
        hi[t], lo[t], _, _ = O.v_thresholds(v[t], 21)
        vlut[t] = O.v_token_lut(vcent, hi[t], lo[t])
    c = torch.zeros((H, W, Lmax), dtype=torch.int32, device=DEV)
    getattr(mod, "vecquant%dappendvecVsparseParallel" % bits)(c, cu(vlut), cu(v.T.reshape(H, 128, T)), cu(lo), cu(hi))
    return dict(vcache=c)


def matvecs(mod, bits):
    from _util import oracle_cache
    L = 700
    c, k, v = oracle_cache(bits, L)
    H, W = 32, 128 * bits // 32
    kc, vc = cu(c.kwords.reshape(H, W, c.Lmax)), cu(c.vwords.reshape(H, W, c.Lmax))
    lut = cu(c.klut["lut"].reshape(H, 128, -1))
    q = cu(O.rope_rotate_q(spec().q_vec(7), L + 3, 10000.0)[None])
    x = np.random.default_rng(bits).standard_normal((1, H, L)).astype(np.float32)
    p = torch.softmax(cu(x) * 2, -1).half().float()
    out = {}
    for sparse in (False, True):
        sfx = "2" if sparse else ""
        m = torch.zeros((1, H, L), device=DEV)
        op = getattr(mod, "vecquant%dmatmul_nuq_perchannel_transposed_rope_mha_batched_fused_opt%s" % (bits, sfx))
        if sparse:
            op(q, kc, m, lut, L, cu(c.k_out), cu(c.k_idx), 10000.0, 3)
        else:
            op(q, kc, m, lut, L, 10000.0, 3)
        o = torch.zeros((1, H, 128), device=DEV)
        op = getattr(mod, "vecquant%dmatmul_nuq_perchannel_transposed_mha_batched_fused_opt%s" % (bits, sfx))
        if sparse:
            op(p, vc, o, cu(c.vlut), L, cu(c.v_out), cu(c.v_idx))
        else:
            op(p, vc, o, cu(c.vlut), L)
        out["k" + sfx], out["v" + sfx] = m, o
    return out


def uncapped_orig_path(mod):
    """Returns (bit-exact results, matvec results)."""
    klut, vcent = quantizer(4)
    sp = spec()
    H, W, Lmax, T = 32, 16, 64, 12
    k, v = sp.k_tokens(T, 51), sp.v_tokens(T, 52)
    lut = cu(klut["lut"].reshape(H, 128, -1))
    lo, hi, zp = cu(klut["thr_lower"]), cu(klut["thr_upper"]), cu(klut["zeropoint"])
    kc = torch.zeros((H, W, Lmax), dtype=torch.int32, device=DEV)
    vc = torch.zeros_like(kc)
    vlut = torch.zeros((Lmax, 16), dtype=torch.float32, device=DEV)
    e = lambda: torch.tensor([]).to(DEV)
    rows, cols, vals, start = e(), e(), e(), e()
    vrows, vcols, vvals, vstart = e(), e(), e(), e()
    for t in range(T):
        rows, cols, vals, start, nth, cnt = mod.vecquant4appendvecKsparseorig(kc, lut, cu(k[t]), zp, rows, cols, vals, start, lo, hi, t)
        thi, tlo, _, _ = O.v_thresholds(v[t], 21)
        lt = O.v_token_lut(vcent, thi, tlo)
        vlut[t] = cu(lt)
        vrows, vcols, vvals, vstart, vnth, vcnt = mod.vecquant4appendvecVsparseorig(
            vc, vlut, cu(v[t]), float(lt[7]), vrows, vcols, vvals, vstart, float(tlo), float(thi), t)
    L = T
    q = cu(O.rope_rotate_q(sp.q_vec(3), L, 10000.0)[None])
    mul = torch.zeros((1, H, L), device=DEV)
    mod.vecquant4matmul_nuq_perchannel_transposed_rope_mha_batched_fused_opt2_orig(
        q, kc, mul, lut, L, rows, cols, start, vals, L, int(nth[0]), int(vals.shape[0]), 10000.0, 0)
    p = torch.softmax(torch.arange(H * L, device=DEV).float().view(1, H, L).sin(), -1)
    out = torch.zeros((1, H, 128), device=DEV)
    mod.vecquant4matmul_nuq_perchannel_transposed_mha_batched_fused_opt2_orig(
        p, vc, out, vlut, L, vrows, vcols, vstart, vvals, L, int(vnth[0]), int(vvals.shape[0]))
    exact = dict(kc=kc, vc=vc, rows=rows, cols=cols, vals=vals, start=start, vrows=vrows, vcols=vcols, vvals=vvals,
                 vstart=vstart, nth=np.array([int(nth[0]), int(vnth[0])], np.int64))
    return exact, dict(mul=mul, out=out)


@pytest.mark.parametrize("bits", [4, 3, 2])
def test_single_token_appends_bit_exact_vs_reference(g, qc, bits):
    assert_bit_exact(g, "appends_b%d" % bits, single_token_appends(qc, bits))


@pytest.mark.parametrize("bits", [4, 2])
def test_prefill_v_packer_bit_exact_vs_reference(g, qc, bits):
    # (3-bit is excluded: the reference kernel indexes the LUT by channel there, quant_cuda_kernel.cu:2574-2579)
    assert_bit_exact(g, "prefill_v_b%d" % bits, prefill_v_packer(qc, bits))


@pytest.mark.parametrize("bits", [4, 3, 2])
def test_matvecs_vs_reference_kernels(g, qc, bits):
    for key, t in matvecs(qc, bits).items():
        assert golden_rel_err(g, "matvecs_b%d" % bits, key, t)[0] < 2e-5, key


def test_uncapped_orig_path_vs_reference(g, qc):
    """vecquant4appendvec{K,V}sparseorig + ..._opt2_orig: CSR/CSC arrays and results identical to the reference."""
    exact, close = uncapped_orig_path(qc)
    assert_bit_exact(g, "orig", exact)
    for key, t in close.items():
        assert golden_rel_err(g, "orig", key, t)[0] < 2e-5, key
