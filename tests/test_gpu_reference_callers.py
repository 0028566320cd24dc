"""GPU: the repository's cache managers (kvquant_b200.cache.QuantK / QuantV) on the drop-in boundary against the
reference's REAL caller code.

The reference's `QuantK` / `QuantV` (modeling_llama.py lines 352-975, 978-1385) are cut verbatim by
oracle/build_ref_py.py and driven by tests/golden/gen_refgpu_golden.py through the reference's own sequence --
load_lookup_table, one prefill `parallel_pack`, then decode steps of `forward_fused_sparse` chained as
modeling_llama.py:1803-1820 and 1963-1999 do (CPU top-k of v, scores.half()/sqrt(d), fp32 softmax -> fp16, V op) --
once on the reference's own CUDA extension and once with `import quant_cuda` resolving to this repository's shim.
Their results are stored in tests/golden/refgpu_callers.npz; here the mirror classes run the same sequence on the shim
and are compared: cache words, per-token LUT rows, outlier rows and indices bit for bit; the fp16 scores and outputs
of a fixed set of decode steps, whole, to fp16 accuracy."""
import math
import warnings

import numpy as np
import pytest
import torch

from _util import assert_bit_exact, golden_pair, load_golden, spec, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
H, HID = 32, 4096
GOLDEN_FILE = "refgpu_callers.npz"
# (prefill tokens, decode steps, Lmax, token seeds, query seed).  REF_EXT: the reference classes on the reference's own
# extension.  Prefill of 32 tokens: the reference's K prefill packer stages its tables in shared memory without a
# barrier (quant_cuda_kernel.cu:1857-1883; 128 threads per block); with more than one warp of tokens its output is not
# reproducible run to run (observed on the B200: 256-320 differing values between two identical calls), so a
# bit-for-bit comparison against it is only meaningful while one warp owns all the tokens.  ON_SHIM: the reference
# classes on this repository's shim.
REF_EXT = (32, 64, 256, (21, 22), 5)
ON_SHIM = (32, 24, 128, (31, 32), 6)
K_PREFILL = ("kcache_prefill", "k_out_idx_prefill", "k_out_prefill")


def _topk_v(v_flat_gpu, kk):
    """modeling_llama.py:1813-1820: top-k of the new value vector on the CPU, results back on the device."""
    v = v_flat_gpu.cpu()
    uv, ui = torch.topk(v, kk)
    lv, li = torch.topk(v, kk, largest=False)
    return uv.cuda(), ui.cuda(), lv.cuda(), li.cuda()


def _drive(QK, QV, bits, cal, k_pre, v_pre, k_dec, v_dec, q_dec, Lmax):
    """One manager pair through prefill + decode; returns (kmgr, vmgr, scores list, outputs list)."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")   # the reference wraps tensors in torch.tensor(...)
        kmgr = QK(bits=bits, hidden_size=HID, num_heads=H, max_position_embeddings=Lmax, include_sparse=True,
                  sparsity_threshold=0.99, rope_theta=10000)
        vmgr = QV(bits=bits, hidden_size=HID, num_heads=H, max_position_embeddings=Lmax, include_sparse=True,
                  sparsity_threshold=0.99)
        kmgr.load_lookup_table(cal["k"], include_sparse=True, sparsity_threshold=0.99)
        vmgr.load_lookup_table(cal["v"], include_sparse=True, sparsity_threshold=0.99)
        kk = int(((1 - 0.99) / 2) * HID) + 2
        T = k_pre.shape[0]
        # prefill (modeling_llama.py:1829-1832, 1907-1927): key_states[0].transpose(1, 2) is [H, 128, T]
        ks = k_pre.view(1, T, H, 128).transpose(1, 2).half()
        vs = v_pre.view(1, T, H, 128).transpose(1, 2).half()
        vf = v_pre.float()
        uv, ui = torch.topk(vf, kk, dim=-1)
        lv, li = torch.topk(vf, kk, dim=-1, largest=False)
        kmgr.parallel_pack(ks[0].transpose(1, 2))
        vmgr.parallel_pack(vs[0].transpose(1, 2), uv, ui, lv, li)
        scores, outs = [], []
        for i in range(k_dec.shape[0]):
            q = q_dec[i].view(H, 1, 128).half()
            kn = k_dec[i].view(1, H, 1, 128).half()
            vn = v_dec[i].view(1, H, 1, 128).half()
            tk = _topk_v(vn.flatten().float(), kk)
            s = kmgr.forward_fused_sparse(q, kn)                               # [H, 1, L] fp16
            scores.append(s.clone())
            a = s.unsqueeze(0) / math.sqrt(128)
            p = torch.nn.functional.softmax(a, dim=-1, dtype=torch.float32).to(torch.float16).squeeze(0)
            o = vmgr.forward_fused_sparse(p, vn, *tk)                          # [H, 1, 128] fp16
            outs.append(o.clone())
    return kmgr, vmgr, scores, outs


def run(QK, QV, bits, case):
    """Drive a manager pair through `case`; returns (bit-exact state split at the prefill, per-step results)."""
    T, ND, Lmax, (ks, vs), qs = case
    sp = spec()
    cal = synth.calibrate(sp, bits, calib_tokens=512, seed=7)
    # fp16-representable inputs: the reference feeds .half() activations to both managers
    k_all = torch.from_numpy(sp.k_tokens(T + ND, seed=ks)).to(DEV).half().float()
    v_all = torch.from_numpy(sp.v_tokens(T + ND, seed=vs)).to(DEV).half().float()
    g = torch.Generator(device=DEV).manual_seed(qs)
    q_dec = torch.randn((ND, H, 128), generator=g, device=DEV)
    km, vm, scores, outs = _drive(QK, QV, bits, cal, k_all[:T], v_all[:T], k_all[T:], v_all[T:], q_dec, Lmax)
    L = T + ND
    assert km.klen == L and vm.vlen == L
    exact = {"k_lut": km.lookup_table.reshape(-1), "v_lut": vm.lookup_table[:L],
             "v_out_idx": vm.outlier_indices[:L], "v_out": vm.outliers[:L]}
    for part, sl in (("prefill", slice(0, T)), ("decode", slice(T, L))):
        exact["kcache_" + part] = km.kcache[:, :, sl]
        exact["k_out_idx_" + part] = km.outlier_indices[sl]
        exact["k_out_" + part] = km.outliers[sl]
        exact["vcache_" + part] = vm.vcache[:, :, sl]
    steps = sorted(set(range(0, ND, 8)) | {ND - 1})
    close = {}
    for i in steps:
        close["scores%d" % i], close["out%d" % i] = scores[i][:, 0], outs[i][:, 0]
    return exact, close


def _compare(g, prefix, exact, close, skip=()):
    assert_bit_exact(g, prefix, {k: t for k, t in exact.items() if k not in skip})
    for key in sorted(close):
        a, b, _, full = golden_pair(g, prefix, key, close[key])
        if key.startswith("scores"):
            # fp16 scores: the fp32 results agree to ~1e-6, so at most an occasional one-ulp rounding flip
            assert np.abs(a - b).max() <= 2.0 ** -10 * max(1.0, full), key
            assert (a == b).mean() > 0.98, key
        elif "out" not in skip:
            assert np.abs(a - b).max() <= 2e-3 * max(full, 1e-3), key


@pytest.mark.parametrize("bits", [4, 3])
def test_mirror_classes_match_the_reference_classes_on_the_reference_extension(bits):
    from kvquant_b200 import cache as kc
    g = load_golden(GOLDEN_FILE)
    exact, close = run(kc.QuantK, kc.QuantV, bits, REF_EXT)
    # The reference's K prefill state is stored only when two runs of its racy packer agreed (see REF_EXT); the file
    # says so explicitly, and the decode-time K state is compared in any case.
    # 3-bit V prefill: the reference kernel indexes the LUT by channel for entries 1..7 (quant_cuda_kernel.cu:2574-2579,
    # a defect our packer does not reproduce, DESIGN.md section 2) -> V codes from the decode-time slots only, and the
    # V outputs differ by that defect too
    skip = ("vcache_prefill", "out") if bits == 3 else ()
    if bool(g["ext_b%d.k_prefill_dropped" % bits]):
        skip += K_PREFILL
    _compare(g, "ext_b%d" % bits, exact, close, skip)


@pytest.mark.parametrize("bits", [4, 3, 2])
def test_mirror_classes_equal_the_reference_classes_on_the_shim(bits):
    """kvquant_b200.cache.QuantK / QuantV (device-side top-k, vectorised LUT build) against the reference's own classes
    on the shim: same caches bit for bit, same fp16 results (same kernels, same inputs)."""
    from kvquant_b200 import cache as kc
    g = load_golden(GOLDEN_FILE)
    exact, close = run(kc.QuantK, kc.QuantV, bits, ON_SHIM)
    _compare(g, "shim_b%d" % bits, exact, close)
