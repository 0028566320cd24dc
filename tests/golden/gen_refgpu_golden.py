#!/usr/bin/env python
"""Generate tests/golden/refgpu_{vs_reference,callers,baseline,fullsize}.npz from the REFERENCE's own code on a GPU.

Needs what oracle/build_ref.py and oracle/build_ref_py.py make from a checkout of the reference project:
oracle/_ref/quant_cuda_ref.so (the unmodified reference extension compiled for sm_100a) and
oracle/_ref/ref_cache_managers.py (its QuantK / QuantV cut verbatim).  Each GPU test that compares against the
reference defines its computation as a function of the boundary module (or manager classes); this script runs those
functions on the reference and stores the results (tests/_util.py: digests of bit-exact results; tolerance-compared
results whole, except the 4K..128K-token score arrays, kept as a fixed sample plus per-row sums and norms over all
elements), so that the tests need neither the reference nor its build.

    python tests/golden/gen_refgpu_golden.py [--out DIR]      # default: tests/golden
"""
import argparse
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import build_ref  # noqa: E402
import build_ref_py  # noqa: E402
from _util import digest, golden_record  # noqa: E402
import test_gpu_baseline_configs as t_base  # noqa: E402
import test_gpu_reference_callers as t_call  # noqa: E402
import test_gpu_vs_reference as t_ref  # noqa: E402
import test_zy_fullsize_properties as t_full  # noqa: E402


def save(out_dir, name, rec):
    path = os.path.join(out_dir, name)
    np.savez_compressed(path, **rec)
    print("wrote", path, os.path.getsize(path), flush=True)
    assert os.path.getsize(path) < 1 << 20, "golden files stay under 1 MB: sample more of the large results"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=HERE)
    out_dir = ap.parse_args().out
    os.makedirs(out_dir, exist_ok=True)
    ref = build_ref.load()
    assert ref is not None and os.path.exists(build_ref_py.OUT), "build oracle/_ref/ from the reference first"
    from kvquant_b200 import quant_cuda as shim
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        on_ref = build_ref_py.load(ref, "ref_managers_on_ref")
        on_shim = build_ref_py.load(shim, "ref_managers_on_shim")

    rec = {}
    for bits in (4, 3, 2):
        rec.update(golden_record("appends_b%d" % bits, exact=t_ref.single_token_appends(ref, bits)))
        rec.update(golden_record("matvecs_b%d" % bits, close=t_ref.matvecs(ref, bits)))
    for bits in (4, 2):
        rec.update(golden_record("prefill_v_b%d" % bits, exact=t_ref.prefill_v_packer(ref, bits)))
    exact, close = t_ref.uncapped_orig_path(ref)
    rec.update(golden_record("orig", exact=exact, close=close))
    save(out_dir, t_ref.GOLDEN_FILE, rec)

    rec = {}
    for bits in (4, 3):
        exact, close = t_call.run(on_ref.QuantK, on_ref.QuantV, bits, t_call.REF_EXT)
        again, _ = t_call.run(on_ref.QuantK, on_ref.QuantV, bits, t_call.REF_EXT)
        racy = [k for k in t_call.K_PREFILL if digest(exact[k]) != digest(again[k])]
        if racy:   # the reference's K prefill packer disagreed with itself: keep its decode-time state only
            print("bits %d: reference K prefill not reproducible (%s); stored without it" % (bits, racy), flush=True)
            for k in t_call.K_PREFILL:
                del exact[k]
        rec.update(golden_record("ext_b%d" % bits, exact=exact, close=close))
        rec["ext_b%d.k_prefill_dropped" % bits] = np.array(bool(racy))
    for bits in (4, 3, 2):
        exact, close = t_call.run(on_shim.QuantK, on_shim.QuantV, bits, t_call.ON_SHIM)
        rec.update(golden_record("shim_b%d" % bits, exact=exact, close=close))
    save(out_dir, t_call.GOLDEN_FILE, rec)

    rec = {}
    for name, bits, H, L, sparse in t_base.CASES:
        lc, q, p = t_base.filled_cache(bits, H, L, sparse)
        rec.update(golden_record(name, close=t_base.legacy_ops(ref, lc, q, p, bits, H, L, sparse, chain=True)))
        del lc
        torch.cuda.empty_cache()
    save(out_dir, t_base.GOLDEN_FILE, rec)

    rec = {}
    for bits in (4, 3):
        lc = t_full.fill(bits)
        rec.update(golden_record("b%d" % bits, close=t_full.legacy_ops(bits, lc, ref)))
        del lc
        torch.cuda.empty_cache()
    save(out_dir, "refgpu_fullsize.npz", rec)


if __name__ == "__main__":
    main()
