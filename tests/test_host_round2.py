"""CPU: host-side logic added in round 2 -- the GPU-free reference arm of bench.py (fixed sample, host-generated cache,
core accounting), the extraction of the reference's QuantK / QuantV source, the oracle's K-outliers-only mode and the
algorithmic-byte figures of the dense-only / K-only workloads (SURVEY.md 8d)."""
import ast
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

from _util import O, quantizer, spec  # noqa: E402


def test_reference_arm_runs_without_a_gpu_and_reports_its_sample():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", KVQ_CPU_SAMPLE_TOKENS="512")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--workload", "7b-4b-32k"], env=env, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-1500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] == line["e2e"]["value"] > 0
    assert "fixed 512 of 32768 tokens" in cb["sample"] and "cgroup cpu quota" in cb["sample"]
    assert cb["worst"] <= cb["median"] <= cb["value"]
    assert line["config"]["workload"] == "7b-4b-32k" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_host_generated_layer_has_the_cache_layout():
    import bench
    for bits, sparse_k, sparse_v in ((4, True, True), (3, True, False), (4, False, False)):
        a = bench.synth_host_layer(bits, 32, 256, 42, sparse_k, sparse_v)
        W = 4096 * bits // 32
        assert a["kcache"].shape == (W, a["Lmax"]) and a["kcache"].dtype == np.int32
        assert a["klut"].shape == (4096, 2 ** bits) and np.all(np.diff(a["klut"], axis=1) >= 0)      # sorted LUT rows
        assert (a["k_out"] is not None) == sparse_k and (a["v_out"] is not None) == sparse_v
        if sparse_k:
            assert a["k_idx"].shape == (a["Lmax"], 42) and np.all(np.diff(a["k_idx"], axis=1) > 0)    # sorted, distinct
            assert a["k_idx"].min() >= 0 and a["k_idx"].max() < 4096
    n, desc = bench.host_cores()
    assert 1 <= n <= len(os.sched_getaffinity(0)) and "affinity" in desc


def test_reference_class_extraction_is_verbatim(tmp_path):
    import build_ref_py
    # a module laid out like the reference's modeling_llama.py: the three wanted definitions among others,
    # a decorator, comments, blank lines and odd spacing that a re-rendering of the AST would not keep
    src_path, out_path = tmp_path / "modeling_llama.py", tmp_path / "_ref" / "ref_cache_managers.py"
    src_path.write_text(
        "import torch\n\nclass LlamaRMSNorm:\n    pass\n\n\n"
        "@torch.no_grad()\ndef compute_lut(x,  y):   # two spaces kept\n    return (x +\n            y)\n\n"
        "def unrelated():\n    return 1\n\n"
        "class QuantK(object):\n    '''doc'''\n\n    def f(self):\n        return 0x10  # hex kept\n\n"
        "X = 3\n\nclass QuantV:\n    a = [1,\n         2]\n")
    assert build_ref_py.build(src=str(src_path), out=str(out_path))
    out = out_path.read_text()
    tree = ast.parse(out)
    names = [n.name for n in tree.body if isinstance(n, (ast.FunctionDef, ast.ClassDef))]
    assert names == ["compute_lut", "QuantK", "QuantV"]
    src = src_path.read_text().splitlines(keepends=True)
    ref_tree = ast.parse("".join(src))
    for node in ref_tree.body:
        if isinstance(node, (ast.FunctionDef, ast.ClassDef)) and node.name in build_ref_py.WANTED:
            first = min([node.lineno] + [d.lineno for d in node.decorator_list])
            assert "".join(src[first - 1:node.end_lineno]) in out      # byte for byte
    assert "unrelated" not in out and "LlamaRMSNorm" not in out
    # the generated file lives in the git-ignored oracle/_ref/ only
    assert os.path.dirname(build_ref_py.OUT).endswith(os.path.join("oracle", "_ref"))
    rc = subprocess.run(["git", "check-ignore", "-q", build_ref_py.OUT], cwd=ROOT).returncode
    assert rc in (0, 128), "oracle/_ref/ref_cache_managers.py must stay out of history"   # 128: not a git checkout


def test_oracle_k_only_mode_is_sparse_k_plus_dense_v():
    bits, H, L = 3, 32, 24
    klut, vcent = quantizer(bits)
    sp = spec()
    k, v = sp.k_tokens(L, 3), sp.v_tokens(L, 4)
    full = O.OracleCache(bits, H, 64, klut, vcent)
    dense = O.OracleCache(bits, H, 64, klut, vcent, include_sparse=False)
    konly = O.OracleCache(bits, H, 64, klut, vcent, include_sparse=True, sparse_v=False)
    for t in range(L):
        for c in (full, dense, konly):
            c.append(k[t], v[t])
    assert np.array_equal(konly.kwords, full.kwords) and np.array_equal(konly.k_out, full.k_out) and np.array_equal(konly.k_idx, full.k_idx)
    assert np.array_equal(konly.vwords, dense.vwords) and np.array_equal(konly.vlut, dense.vlut)
    assert not np.array_equal(dense.vlut[:L], full.vlut[:L])      # min/max range vs 22nd order statistics
    q = O.rope_rotate_q(sp.q_vec(1), L, 10000.0)
    p = np.full((H, L), 1.0 / L, np.float32)
    assert np.allclose(konly.k_scores(q), full.k_scores(q)) and np.allclose(konly.v_output(p), dense.v_output(p))


def test_algorithmic_bytes_of_the_1m_workloads_match_the_survey():
    from kvquant_b200 import decode as kd
    # SURVEY.md 8d: 7B 4-bit dense-only 4160 B/token; 13B 3-bit + capped-K only 3840 + 416 + 32 = 4288
    c3 = kd.DecodeConfig.llama7b(bits=4, include_sparse=False)
    c4 = kd.DecodeConfig.llama13b(bits=3, include_sparse=True, sparse_v=False)
    assert kd.layer_step_bytes(c3, 1) == 4160 and kd.layer_step_bytes(c4, 1) == 4288
    assert kd.layer_step_bytes(kd.DecodeConfig.llama7b(bits=4), 1) == 4832
    assert kd.layer_step_bytes(kd.DecodeConfig.llama7b(bits=3), 1) == 3776
