"""GPU: parity at BASELINE.json's config sizes against the REFERENCE's own CUDA kernels.

  configs[0]  single layer, 4-bit, 4K tokens, with and without 1 % outliers
  configs[1]  LLaMA-7B shapes, 4-bit + 1 % outliers, 32K tokens
  13B shapes  (H = 40, 52 outlier columns), 3-bit, 8K tokens  -- the shape of configs[4] at a size the reference op
              chain finishes in milliseconds

Caches are filled by the real prefill packers (synth.fill_layer_cache_gpu, seeded); the reference's results on the
same caches (oracle/_ref/quant_cuda_ref.so, the unmodified reference extension) are stored in
tests/golden/refgpu_baseline.npz by tests/golden/gen_refgpu_golden.py -- the [H, 128] outputs whole, the K scores as a
fixed sample of 16384 elements plus per-head sums and norms over all of them (tests/_util.py):
  * our legacy K / V ops vs the reference's kernels: norm-wise <= 2e-5 AND per head (every head relative to that head's
    own largest value) <= 1e-4 -- a wrong small element cannot hide behind a large one in another head -- AND every
    head's sum and norm of the K scores within 2e-5;
  * the fused attend (exact tables, the default) vs the reference op chain K op -> softmax -> V op: <= 1e-4 / per head
    3e-4; with fp16 tables: <= 2e-3 / per head 1e-2 (DESIGN.md section 5 for where that error comes from)."""
import numpy as np
import pytest
import torch

from _util import golden_rel_err, load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN_FILE = "refgpu_baseline.npz"

CASES = [  # (name, bits, H, L, sparse)
    ("configs0-4b-4k-dense", 4, 32, 4096, False),
    ("configs0-4b-4k-sparse", 4, 32, 4096, True),
    ("configs1-7b-4b-32k", 4, 32, 32768, True),
    ("13b-3b-8k", 3, 40, 8192, True),
]


def filled_cache(bits, H, L, sparse):
    """(layer cache of L synthetic tokens, query [1, H, 128], V-op weights [1, H, L])."""
    from kvquant_b200 import synth, cache as kc
    sp = synth.SynthSpec(H, 128, seed=0)
    cal = synth.calibrate(sp, bits, calib_tokens=512, seed=7)
    klut = kc.build_k_lookup_table(cal["k"][0], cal["k"][1], cal["k"][2][0], H, device=DEV)
    lc = kc.LayerCache.from_luts(bits, H, L + 64, dict(lut=klut["lut"], lut2=None, thr_lower=klut["thr_lower"],
                                                      thr_upper=klut["thr_upper"]), cal["v"][2][0], device=DEV,
                                 include_sparse=sparse)
    synth.fill_layer_cache_gpu(lc, sp, L, seed=bits + H)
    g = torch.Generator(device=DEV).manual_seed(L + H)
    q = torch.randn((1, H, 128), generator=g, device=DEV).half().float()
    x = np.random.default_rng(L + H).standard_normal((1, H, L)).astype(np.float32)
    p = torch.softmax(torch.from_numpy(x).to(DEV) * 2, -1).contiguous()
    return lc, q, p


def legacy_ops(mod, lc, q, p, bits, H, L, sparse, chain=False):
    """K op scores [H, L], V op output [H, 128] for the weights p, and with chain=True the op chain
    K op -> softmax -> V op [H, 128]."""
    sfx = "2" if sparse else ""
    kop = getattr(mod, "vecquant%dmatmul_nuq_perchannel_transposed_rope_mha_batched_fused_opt%s" % (bits, sfx))
    vop = getattr(mod, "vecquant%dmatmul_nuq_perchannel_transposed_mha_batched_fused_opt%s" % (bits, sfx))
    lutK = lc.klut.view(H, 128, -1)

    def v_op(w):
        mul = torch.zeros((1, H, 128), device=DEV)
        if sparse:
            vop(w, lc.vcache, mul, lc.vlut, L, lc.v_outliers, lc.v_outlier_idx)
        else:
            vop(w, lc.vcache, mul, lc.vlut, L)
        return mul[0]

    s = torch.zeros((1, H, L), device=DEV)
    if sparse:
        kop(q, lc.kcache, s, lutK, L, lc.k_outliers, lc.k_outlier_idx, 10000.0, 0)
    else:
        kop(q, lc.kcache, s, lutK, L, 10000.0, 0)
    out = {"k": s[0], "v": v_op(p)}
    if chain:
        out["chain"] = v_op(torch.softmax(s[0] / np.sqrt(128), -1)[None].contiguous())
    return out


@pytest.mark.parametrize("name,bits,H,L,sparse", CASES, ids=[c[0] for c in CASES])
def test_ops_and_fused_attend_vs_reference_kernels(name, bits, H, L, sparse):
    from kvquant_b200 import quant_cuda as qc
    g = load_golden(GOLDEN_FILE)
    lc, q, p = filled_cache(bits, H, L, sparse)
    for key, t in legacy_ops(qc, lc, q, p, bits, H, L, sparse).items():
        e_norm, e_head, e_sums = golden_rel_err(g, name, key, t)
        assert e_norm < 2e-5 and e_head < 1e-4 and e_sums < 2e-5, (key, e_norm, e_head, e_sums)
    for precision, tol, tol_head in (("fp32", 1e-4, 3e-4), ("fp16", 2e-3, 1e-2)):
        lc.precision = precision
        e_norm, e_head, _ = golden_rel_err(g, name, "chain", lc.attend(q[0].contiguous()))   # stored whole
        assert e_norm < tol and e_head < tol_head, (precision, e_norm, e_head)
