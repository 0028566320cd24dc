#!/usr/bin/env python
"""bench.py -- decode tokens/sec of a LLaMA-7B-shaped model over the quantised KV cache (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W [--workload NAME] [--impl reference] [--dump-outputs DIR]

A "step" is one batch-1 decode step at cache length L of the named workload: for every layer q/k/v projection,
fused device-side append (NUQ quantise + top-K outlier split + pack), fused attend over the packed cache
(LUT dequant + outlier SpMV + RoPE + softmax + V), o_proj and MLP, then norm + lm_head.  Weights are random-init
fp16 of the LLaMA architecture, caches are filled with synthetic K/V through the real prefill packers.
The whole step is one CUDA graph; replays re-run the step at the SAME cache length (the fused append overwrites
its slot), so all K timed steps are measured at the named seqlen.

N > 1, one process per GPU under torch.distributed / NCCL, two layouts (--parallelism):
  pp  layer-group pipeline -- the reference's own multi-GPU scheme (modeling_llama.py:2428-2453) and what north_star
      prescribes: NCCL send/recv of the [hidden] fp16 vector over NVLink.  At batch 1 the stages run one after
      another, so it buys capacity (1M-token contexts), not tokens/sec.
  sp  sequence-sharded attention (SURVEY 8e-2 / 8f-1): weights replicated, every rank holds 1/N of every layer's
      cache, per layer one all-gather of the partial (out, lse) results (H*129 floats per rank) and a merge kernel.
      This is the layout in which decode speeds up with N; it is the default ("auto") when the workload divides.
Both are strong scaling of the same fixed workload ("scaling": "strong").

--impl reference: the reference's CPU implementation of the path, i.e. the C port of the kernel semantics
(oracle/kvq_oracle_port.c; /root/reference does not exist on the GPU box and the reference's CPU path is Python)
timed on the host cores over a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark writes nothing into the tree it runs from: without this, its first import of modules that build()
# does not import (kvquant_b200.decode, .synth, .p2p) would add __pycache__/ files there
sys.dont_write_bytecode = True

WORKLOADS = {
    # name: (model, bits, L (quantised slots), n_sink, outliers, description = BASELINE.json configs[i])
    #   outliers: "kv" = 1 % dense-and-sparse on K and V, "k" = capped K outliers only, "none" = dense-only
    "7b-3b-128k": ("7b", 3, 131072, 5, "kv", "LLaMA-7B 3b NUQ + 1% outliers + 5 fp16 sink tokens, seqlen 128K, 1xB200 (configs[2])"),
    "7b-4b-128k": ("7b", 4, 131072, 0, "kv", "LLaMA-7B 4b NUQ + 1% outliers, seqlen 128K (north_star roofline target)"),
    "7b-4b-32k": ("7b", 4, 32768, 0, "kv", "LLaMA-7B 4b NUQ + 1% outliers, seqlen 32K, 1xB200 decode (configs[1])"),
    "7b-4b-4k": ("7b", 4, 4096, 0, "kv", "single-node smoke size"),
    "7b-4b-1m": ("7b", 4, 1048576, 0, "none", "LLaMA-7B 4b NUQ, seqlen 1M, layer-pipeline across 4xB200 (configs[3])"),
    "13b-3b-1m": ("13b", 3, 1048576, 0, "k", "LLaMA-13B 3b NUQ + capped-K outliers, seqlen 1M, layer-pipeline across 8xB200 (configs[4])"),
}
DEFAULT_WORKLOAD = "7b-3b-128k"   # BASELINE.json's metric is quoted at seqlen 128K; this config fits one GPU


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def build_quantizer(cfg_bits, H, device):
    from kvquant_b200 import synth, cache as kc
    sp = synth.SynthSpec(H, 128, seed=0)
    cal = synth.calibrate(sp, cfg_bits, calib_tokens=512, seed=7)
    t = kc.build_k_lookup_table(cal["k"][0], cal["k"][1], cal["k"][2][0], H, device=device)
    klut = dict(lut=t["lut"], lut2=None, thr_lower=t["thr_lower"], thr_upper=t["thr_upper"])
    return sp, dict(klut=klut, v_cent=cal["v"][2][0])


# ------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: CPU port of the path on the host cores, fixed bounded sample, no GPU involved
# ------------------------------------------------------------------------------------------------------------
# tokens of ONE layer per timed call (fixed: the same work on every box and every run; the override is for the tests)
CPU_SAMPLE_TOKENS = int(os.environ.get("KVQ_CPU_SAMPLE_TOKENS", "32768"))


def host_cores():
    """(usable cores, description): scheduler affinity and the cgroup CPU quota, whichever is smaller."""
    n_aff = len(os.sched_getaffinity(0))
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            a, b = f.read().split()[:2]
            if a != "max":
                quota = float(a) / float(b)
    except (OSError, ValueError):
        pass
    n = n_aff if quota is None else max(1, min(n_aff, int(quota)))
    return n, "affinity %d cores, cgroup cpu quota %s" % (n_aff, "none" if quota is None else "%.1f cores" % quota)


def synth_host_layer(bits, H, Ls, n_out, sparse_k, sparse_v, seed=0):
    """One layer's quantised cache of Ls tokens generated ON THE HOST (numpy): uniformly random codes, a calibrated
    K LUT, per-token V LUT rows, sorted distinct outlier indices with heavy-tailed values.  The C port's run time does
    not depend on the code values (same loads, same arithmetic), so this times exactly the work of a real cache."""
    import numpy as np
    from kvquant_b200 import synth
    rng = np.random.default_rng(seed)
    hidden = H * 128
    W = hidden * bits // 32
    Lmax = Ls + 64
    sp = synth.SynthSpec(H, 128, seed=0)
    cal = synth.calibrate(sp, bits, calib_tokens=256, seed=7)
    up = cal["k"][0].astype(np.float16).astype(np.float32)
    lo = cal["k"][1].astype(np.float16).astype(np.float32)
    cent = np.sort(cal["k"][2][0].ravel().astype(np.float32))
    klut = (cent[None, :] * ((up - lo) / 2)[:, None] + ((up + lo) / 2)[:, None]).astype(np.float32)
    vcent = np.sort(cal["v"][2][0].ravel().astype(np.float32))
    sf = np.exp(rng.normal(0, 0.3, (Lmax, 1))).astype(np.float32) * 2.5
    vlut = (vcent[None, :] * sf + rng.normal(0, 0.05, (Lmax, 1)).astype(np.float32)).astype(np.float32)
    a = dict(kcache=rng.integers(0, 2 ** 32, (W, Lmax), dtype=np.uint32).view(np.int32),
             vcache=rng.integers(0, 2 ** 32, (W, Lmax), dtype=np.uint32).view(np.int32),
             klut=np.ascontiguousarray(klut), vlut=np.ascontiguousarray(vlut), q=sp.q_vec(1), Lmax=Lmax)

    def rows():
        idx = np.sort(np.argsort(rng.random((Lmax, hidden)), axis=1)[:, :n_out], axis=1).astype(np.int32)
        val = rng.standard_t(3, (Lmax, n_out)).astype(np.float32) * 3
        return np.ascontiguousarray(val), np.ascontiguousarray(idx)
    a["k_out"], a["k_idx"] = rows() if sparse_k else (None, None)
    a["v_out"], a["v_idx"] = rows() if sparse_v else (None, None)
    return a


def cpu_baseline_run(bits, H, L, n_out, sparse_k, sparse_v, n_layers, theta, pos_offset, repeats=5, arrays=None):
    """Time the C port's attend (oracle/kvq_oracle_port.c, OpenMP on every usable host core) for one layer over a FIXED
    sample of CPU_SAMPLE_TOKENS tokens, `repeats` times; the best time is extrapolated to tokens/sec of the whole
    model's attention (n_layers x L tokens; the dense GEMVs are NOT added, which only favours the CPU number).
    Returns (tokens_per_sec, cores, sample description, per-call seconds list, arrays)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import build_oracle_c
    lib = build_oracle_c.load()
    cores, cores_desc = host_cores()
    lib.kvq_port_set_threads(cores)        # not OMP_NUM_THREADS (torchrun sets it to 1)
    cores = lib.kvq_port_threads()
    Ls = min(L, CPU_SAMPLE_TOKENS)
    a = arrays if arrays is not None else synth_host_layer(bits, H, Ls, n_out, sparse_k, sparse_v)
    q = np.ascontiguousarray(a["q"], dtype=np.float32)
    out = np.zeros((H, 128), np.float32)
    scratch = np.zeros((H, Ls), np.float32)

    def ptr(x):
        return x.ctypes.data if x is not None else None
    # the port takes one outlier width: rows of a dense-only side are simply absent (NULL)
    times = []
    for _ in range(repeats + 1):
        t0 = time.perf_counter()
        lib.kvq_port_attend(bits, q.ctypes.data, a["kcache"].ctypes.data, a["klut"].ctypes.data, ptr(a["k_out"]),
                            ptr(a["k_idx"]), a["vcache"].ctypes.data, a["vlut"].ctypes.data, ptr(a["v_out"]),
                            ptr(a["v_idx"]), n_out, H, a["Lmax"], Ls, theta, pos_offset, out.ctypes.data,
                            scratch.ctypes.data)
        times.append(time.perf_counter() - t0)
    times = times[1:]                      # first call: page faults / thread start-up
    best = min(times)
    tok_s = 1.0 / (best * (L / Ls) * n_layers)
    desc = ("C port (oracle/kvq_oracle_port.c, OpenMP, %d threads; %s) of one layer's attend over a fixed %d of %d "
            "tokens of a host-generated cache, best of %d calls (%.1f..%.1f ms), extrapolated to %d layers x %d tokens; "
            "GEMVs excluded" % (cores, cores_desc, Ls, L, len(times), 1e3 * best, 1e3 * max(times), n_layers, L))
    return tok_s, cores, desc, times, a


def _time_cuda(fn, iters, warm=2):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def reference_cuda_anchor(lc, cfg, L, n_sink, bits, ms_ours, peak):
    """The kernel-vs-kernel anchor (SURVEY 2.2 / 8d): the reference's OWN CUDA kernels (oracle/_ref/quant_cuda_ref.so =
    deployment/kvquant/quant_cuda_kernel.cu compiled unmodified for sm_100a by oracle/build_ref.py) on this GPU, on one
    layer's cache of this workload: its K op (dense + SPMV_ATOMIC_ROPE_BALANCED) and V op (dense + SPMV_ATOMIC_BALANCED)
    -- the two launches of the chain modeling_llama.py:1963-1999, without its torch glue -- next to our fused attend."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import build_ref
        ref = build_ref.load()
    except Exception as e:  # noqa: BLE001
        ref = None
        why = repr(e)[:120]
    if ref is None:
        return {"unavailable": "oracle/_ref/quant_cuda_ref.so not present (%s)" % (locals().get("why", "not built"))}
    if not (lc.sparse_k and lc.sparse_v):
        return {"unavailable": "the reference has no mixed / dense-only fused op chain to time for this workload"}
    H, dev = cfg.n_heads, lc.device
    q1 = torch.randn((1, H, 128), device=dev).half().float()
    mulK = torch.zeros((1, H, L), device=dev)
    pV = torch.softmax(torch.randn((1, H, L), device=dev), -1)
    mulV = torch.zeros((1, H, 128), device=dev)
    kop = getattr(ref, "vecquant%dmatmul_nuq_perchannel_transposed_rope_mha_batched_fused_opt2" % bits)
    vop = getattr(ref, "vecquant%dmatmul_nuq_perchannel_transposed_mha_batched_fused_opt2" % bits)
    lutK = lc.klut.view(H, 128, -1)
    ms_k = _time_cuda(lambda: kop(q1, lc.kcache, mulK, lutK, L, lc.k_outliers, lc.k_outlier_idx, cfg.rope_theta, n_sink), 5)
    ms_v = _time_cuda(lambda: vop(pV, lc.vcache, mulV, lc.vlut, L, lc.v_outliers, lc.v_outlier_idx), 5)
    nbytes = L * lc.bytes_per_token()
    chain = ms_k + ms_v
    return {"k_op_ms": ms_k, "v_op_ms": ms_v, "chain_ms": chain, "gbs": nbytes / chain / 1e6,
            "frac": nbytes / chain / 1e6 / peak, "ours_ms": ms_ours, "speedup": chain / ms_ours,
            "what": "reference quant_cuda kernels (unmodified, sm_100a) on one layer of this workload, same GPU, same cache"}


def north_star_anchor(dev, cfg7b_like, peak, L=131072, n_caches=3):
    """north_star's roofline kernel: the fused 4-bit NUQ dequant + sparse attend matvec at seqlen 128K (7B shapes,
    1 % outliers), timed with CUDA events while cycling over `n_caches` distinct layer caches (1.8 GB: nothing stays
    in L2), whatever workload this bench run is on."""
    import torch
    from kvquant_b200 import synth
    from kvquant_b200.cache import LayerCache
    H = 32
    sp, quantizer = build_quantizer(4, H, dev)
    caches = []
    for i in range(n_caches):
        lc = LayerCache.from_luts(4, H, L + 64, quantizer["klut"], quantizer["v_cent"], device=dev)
        synth.fill_layer_cache_gpu(lc, sp, L, seed=900 + i)
        caches.append(lc)
    q = torch.randn((H, 128), device=dev).half().float()
    out = {}
    for prec in ("fp16", "fp32"):
        for lc in caches:
            lc.precision = prec

        def run():
            for lc in caches:
                lc.attend(q)
        ms = _time_cuda(run, 10) / n_caches
        nbytes = L * caches[0].bytes_per_token()
        out[prec] = {"ms": ms, "gbs": nbytes / ms / 1e6, "frac": nbytes / ms / 1e6 / peak}
    rec = dict(out["fp16"], workload="7b-4b-128k", algorithmic_bytes_per_launch=L * caches[0].bytes_per_token(),
               table_precision="fp16", exact_fp32_tables=out["fp32"])
    del caches
    torch.cuda.empty_cache()
    return rec


def ncu_traffic(bits, L):
    """dram__bytes_read.sum + dram__bytes_write.sum of one fused attend (all its kernels), per launch, from the
    committed ncu --set full capture of the same shape (profiles/ncu_traffic.json); None when no capture matches."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            for e in json.load(f)["entries"]:
                if e["bits"] == bits and abs(e["L"] - L) <= 1024:
                    return e["dram_bytes_per_launch"]
    except (OSError, KeyError, ValueError):
        pass
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-anchors", action="store_true",
                    help="skip the two extra roofline records (reference CUDA kernels on this GPU, 4-bit 128K attend)")
    ap.add_argument("--parallelism", default="auto", choices=["auto", "pp", "sp"],
                    help="N>1: pp = layer-group pipeline (the reference's scheme, north_star: buys capacity, not "
                         "tokens/sec at batch 1); sp = sequence-sharded attention with replicated weights (SURVEY 8e-2 / "
                         "8f-1: the layout in which decode speeds up with N).  auto = sp when the workload fits, else pp")
    ap.add_argument("--graph", default="dynamic", choices=["dynamic", "static"],
                    help="dynamic: cache length / position live on the device and every replay is the NEXT decode step "
                         "(growing cache); static: every replay re-runs the step at the captured length")
    ap.add_argument("--sp-exchange", default="p2p", choices=["nccl", "p2p"],
                    help="sp only: how the per-GPU partial attention results meet -- p2p (default): ONE kernel per layer "
                         "stores the 16.6 KB partial straight into the peers' IPC-mapped buffers over NVLink, waits for "
                         "theirs and merges (validated against NCCL at 2/4/8 GPUs, tests/test_zz_p2p_exchange.py); "
                         "nccl: all_gather + merge kernel")
    ap.add_argument("--torch-profile", default="", help="write a per-kernel table of 3 graph replays to this file (diagnostic)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the logits the last timed step returned to the host as "
                         "DIR/logits.npy (float32); weights, caches and tokens are seeded, so the same arguments "
                         "give the same inputs and two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the decode step's logits: it needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    import numpy as np
    import torch
    import torch.distributed as dist
    from kvquant_b200 import decode as kd, synth, _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    model, bits, L, n_sink, outl, desc = WORKLOADS[args.workload]
    metric = "decode tokens/sec @ seqlen %dK (LLaMA-%s, bs1)" % (L // 1024, model.upper())
    base = {"metric": metric, "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (random-init fp16 LLaMA-%s weights, synthetic K/V packed by the real prefill packers)" % model.upper()}

    if args.impl == "reference":
        if rank != 0:
            return 0
        dev = torch.device("cpu")        # the reference arm never touches a GPU
    else:
        torch.cuda.set_device(local)
        dev = torch.device("cuda", local)
    if world > 1 and args.impl == "ours":
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    par = args.parallelism
    if par == "auto":
        par = "sp" if (world > 1 and L % world == 0) else "pp"
    par_label = ("sp%d" if (par == "sp" and world > 1) else "pp%d") % world
    if args.impl == "reference":
        par = "pp"          # the CPU arm runs the whole job (all L tokens, all layers) on rank 0's host cores
    sp_mode = (par == "sp" and world > 1)
    if sp_mode and L % world:
        raise SystemExit("sp needs seq_len divisible by the number of GPUs")
    L_local = L // world if sp_mode else L
    # room for every step this run appends (warm-up + profile + timed, device and e2e loops)
    headroom = (2 * (args.steps + args.warmup) + 3 + 8 + 63) // 64 * 64
    mk = kd.DecodeConfig.llama13b if model == "13b" else kd.DecodeConfig.llama7b
    cfg = mk(bits=bits, n_sink=n_sink, max_len=L_local + headroom, include_sparse=(outl != "none"),
             sparse_v=(outl == "kv"))
    sp, quantizer = (None, None) if args.impl == "reference" else build_quantizer(bits, cfg.n_heads, dev)
    config = {"workload": args.workload, "description": desc, "bits": bits, "seq_len": L + n_sink, "n_sink": n_sink,
              "outliers": {"kv": "1% (n_each + n_each per token per cache)", "k": "capped 1% on K only", "none": "none (dense-only)"}[outl],
              "layers": cfg.n_layers, "parallelism": par_label,
              "l2_policy": "inputs larger than L2: every step streams all layers' caches (>= 4 GB) and 13.5 GB of weights",
              "step": ("one CUDA-graph replay = the next decode step of a growing cache (length and position live in "
                       "device memory; step i appends slot L+i and attends over L+i+1 slots)") if args.graph == "dynamic"
              else "one CUDA-graph replay of a full decode step at fixed cache length"}

    # ---------------------------------------------------------------------------------------------------------
    if args.impl == "reference":
        # GPU-free: host-generated cache, fixed sample; one "step" = one timed call of the C port
        n_out = 2 * (int(((1 - 0.99) / 2) * cfg.hidden) + 1)
        tok_s, cores, sample, times, _ = cpu_baseline_run(bits, cfg.n_heads, L, n_out, outl != "none", outl == "kv",
                                                          cfg.n_layers, cfg.rope_theta, n_sink,
                                                          repeats=args.warmup + args.steps)
        timed = times[args.warmup:] if len(times) > args.warmup else times
        Ls = min(L, CPU_SAMPLE_TOKENS)
        vals = sorted(1.0 / (t * (L / Ls) * cfg.n_layers) for t in timed)
        v = vals[-1]                     # best call: the least disturbed one (the host cores are shared)
        line = dict(base, impl="reference", value=v, ms_per_step=1000.0 / v, config=config, gpu_launches=0,
                    cpu_baseline={"value": v, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample,
                                  "median": vals[len(vals) // 2], "worst": vals[0]},
                    e2e={"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                    clocks=None, roofline=None)
        print(json.dumps(line), flush=True)
        return 0

    # ---------------------------------------------------------------------------------------------------------
    sp_exchange = None
    if sp_mode:
        lo, hi = 0, cfg.n_layers
        stage = kd.DecoderStage(cfg, lo, hi, dev, quantizer, seed=0, with_head=True, sp=(rank, world))
        stage.global_pos = n_sink + L
        sp_exchange = "nccl all_gather + merge kernel"
        if args.sp_exchange == "p2p":
            from kvquant_b200.p2p import PeerExchange
            try:
                stage.xchg = PeerExchange(rank, world, cfg.n_heads, dev)
                sp_exchange = "peer-memory stores over NVLink fused with the merge (kvq_attend_exchange_merge)"
            except Exception as e:  # noqa: BLE001  (no peer access / IPC: fall back to the NCCL path on every rank)
                stage.xchg = None
                sp_exchange += " (peer exchange unavailable: %s)" % repr(e)[:80]
            ok = torch.tensor([1 if stage.xchg is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                stage.xchg = None
            else:
                # self-test on this box before anything is captured: 16 exchanges of random partials against
                # all_gather + kvq_attend_merge (tests/_p2p_check.py does 200); any rank unhappy -> every rank uses NCCL
                n = cfg.hidden + cfg.n_heads
                good = 1
                for it in range(16):
                    part = torch.randn(n, device=dev)
                    gath = torch.empty(world * n, device=dev)
                    dist.all_gather_into_tensor(gath, part)
                    want = torch.empty(cfg.hidden, device=dev)
                    _lib.check(_lib.load().kvq_attend_merge(gath.data_ptr(), world, cfg.n_heads, want.data_ptr(),
                                                            torch.cuda.current_stream().cuda_stream))
                    got = torch.empty(cfg.hidden, device=dev)
                    stage.xchg.exchange_merge(part, got)
                    torch.cuda.synchronize()
                    if stage.xchg.failed() or not torch.isfinite(got).all() or (got - want).abs().max().item() > 1e-5 * max(1.0, want.abs().max().item()):
                        good = 0          # (no early exit: the ranks must stay in lockstep through the collectives)
                ok = torch.tensor([good], device=dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                if int(ok.item()) == 0:
                    stage.xchg = None
                    sp_exchange = "nccl all_gather + merge kernel (peer exchange failed its self-test on this box)"
    else:
        lo, hi = kd.partition_layers(cfg.n_layers, world, rank)
        stage = kd.DecoderStage(cfg, lo, hi, dev, quantizer, seed=0, with_head=(rank == 0))
    t_fill = time.time()
    for i, ly in enumerate(stage.layers):
        if sp_mode:
            ly.cache.pos_base = rank * L_local
        synth.fill_layer_cache_gpu(ly.cache, sp, L_local, seed=(lo + i) * 16 + (rank if sp_mode else 0))
    torch.cuda.synchronize()
    t_fill = time.time() - t_fill

    n0 = _lib.launch_count()
    pp_mode = world > 1 and not sp_mode
    gs = kd.GraphedStage(stage, L_local, first=(rank == 0 or sp_mode), last_to_logits=(world == 1 or sp_mode),
                         dynamic=(args.graph == "dynamic"), pos=(n_sink + L) if sp_mode else None,
                         pp=(rank, world) if pp_mode else None)
    launches_per_step = (_lib.launch_count() - n0) // (5 if (sp_mode or pp_mode) else 3)   # eager warm-up passes + 1 capture pass
    pinned_tok = torch.zeros(1, dtype=torch.long).pin_memory()
    pinned_logits = torch.zeros(cfg.vocab, dtype=torch.float16).pin_memory()
    logits_dev = [None]

    def step_device():
        """one decode step, inputs resident on the device"""
        # pp: the hops are NCCL send/recv kernels inside the captured graphs (rank 0 replays two: its layers, then
        # recv + norm + lm_head)
        gs.replay()
        if rank == 0 or sp_mode:
            logits_dev[0] = gs.logits

    def step_e2e(i):
        """same step through host buffers: token id H2D from pinned memory, logits D2H to pinned memory"""
        if rank == 0 or sp_mode:
            pinned_tok[0] = (17 * i + 3) % cfg.vocab
            gs.tok.copy_(pinned_tok, non_blocking=True)
        step_device()
        if rank == 0 or sp_mode:
            pinned_logits.copy_(logits_dev[0], non_blocking=True)
            torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            fn(i)
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for i in range(args.warmup):
        step_device()
    if args.torch_profile and rank == 0:
        from torch.profiler import profile, ProfilerActivity
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(3):
                step_device()
            torch.cuda.synchronize()
        with open(args.torch_profile, "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40, max_name_column_width=90))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total = timed(lambda i: step_device(), args.steps)
    for i in range(args.warmup):
        step_e2e(i)
    ms_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the last timed step is step_e2e(steps - 1): its logits sit in pinned host memory, synchronised
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "logits.npy"), pinned_logits.float().numpy())
    if sp_mode and stage.xchg is not None:
        bad = torch.tensor([1 if stage.xchg.failed() else 0], device=dev)
        dist.all_reduce(bad, op=dist.ReduceOp.MAX)
        if int(bad.item()):
            raise SystemExit("peer-memory exchange timed out on some rank: results invalid (rerun with --sp-exchange nccl)")
    ms_step = ms_total / args.steps
    value = 1000.0 / ms_step
    e2e_value = 1000.0 / (ms_e2e / args.steps)

    # ---- roofline of the dominant op (fused attend), measured live on this stream, cycling over the layers -------
    roof = None
    cpu_b = None
    layers = stage.layers
    q = torch.randn((cfg.n_heads, 128), device=dev).half().float()
    reps = max(2, 64 // len(layers))

    def time_loop(fn):
        for ly in layers[:2]:
            fn(ly)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            for ly in layers:
                fn(ly)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / (reps * len(layers))

    Lq = layers[0].cache.len      # current length (the timed steps appended to the cache)
    # every rank times the fused attend of ITS layers (pp: one record per pipeline stage; sp: per sequence shard)
    ms_att = time_loop(lambda ly: ly.cache.attend(q, rope_theta=cfg.rope_theta))
    ms_all = torch.tensor([ms_att], device=dev)
    if world > 1:
        gath = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(gath, ms_all)
        ms_all = torch.cat(gath)
    if rank == 0:
        peak, peak_src = measured_peak()
        n_out = layers[0].cache.n_out
        b_att = kd.layer_step_bytes(cfg, Lq)
        per_kernel = None
        if outl == "kv":       # the legacy two-op surface (what the reference's QuantK / QuantV call), timed separately
            from kvquant_b200 import quant_cuda as qc
            mulK = torch.zeros((1, cfg.n_heads, Lq), device=dev)
            pV = torch.softmax(torch.randn((1, cfg.n_heads, Lq), device=dev), -1)
            mulV = torch.zeros((1, cfg.n_heads, 128), device=dev)
            q1 = q[None].contiguous()
            kop = getattr(qc, "vecquant%dmatmul_nuq_perchannel_transposed_rope_mha_batched_fused_opt2" % bits)
            vop = getattr(qc, "vecquant%dmatmul_nuq_perchannel_transposed_mha_batched_fused_opt2" % bits)
            ms_k = time_loop(lambda ly: kop(q1, ly.cache.kcache, mulK, ly.cache.klut.view(cfg.n_heads, 128, -1), Lq,
                                            ly.cache.k_outliers, ly.cache.k_outlier_idx, cfg.rope_theta, n_sink))
            ms_v = time_loop(lambda ly: vop(pV, ly.cache.vcache, mulV, ly.cache.vlut, Lq, ly.cache.v_outliers,
                                            ly.cache.v_outlier_idx))
            b_k = Lq * (cfg.hidden * bits // 8 + 8 * n_out)
            b_v = Lq * (cfg.hidden * bits // 8 + 8 * n_out + 4 * 2 ** bits)
            per_kernel = {"legacy_k_op": {"ms": ms_k, "bytes": b_k, "gbs": b_k / ms_k / 1e6, "frac": b_k / ms_k / 1e6 / peak},
                          "legacy_v_op": {"ms": ms_v, "bytes": b_v, "gbs": b_v / ms_v / 1e6, "frac": b_v / ms_v / 1e6 / peak}}
            del mulK, pV
        ach = b_att / ms_att / 1e6
        roof = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": ncu_traffic(bits, Lq),
                "peak_source": peak_src,
                "kernel": "kvq_attend = attend_init + k_outlier_pers + k_scores(3) + v_native + attend_combine",
                "algorithmic_bytes_per_launch": b_att, "ms_per_launch": ms_att,
                "per_kernel": per_kernel,
                "per_rank": [{"rank": r, "ms_per_launch": float(m), "gbs": b_att / float(m) / 1e6,
                              "frac": b_att / float(m) / 1e6 / peak} for r, m in enumerate(ms_all.tolist())],
                "attend_share_of_step": ms_att * len(layers) / ms_step}
        prec = layers[0].cache.precision
        k_names = ("k_ratio_prep", "k_ratio") if prec == "fp32" else ("k_fast_prep", "k_fast")
        roof["kernel"] = ("kvq_attend (table precision %s) = attend_init + %s + [memset + k_outlier_pers] + %s + v_native + "
                          "attend_combine" % (prec, k_names[0], k_names[1]))
        if not args.no_anchors:
            roof["reference_cuda"] = reference_cuda_anchor(layers[0].cache, cfg, Lq, n_sink, bits, ms_att, peak)
            roof["north_star_kernel"] = north_star_anchor(dev, cfg, peak)
        if not args.no_cpu_baseline:
            tok_s, cores, sample, _, _ = cpu_baseline_run(bits, cfg.n_heads, L, n_out, outl != "none", outl == "kv",
                                                          cfg.n_layers, cfg.rope_theta, n_sink, repeats=5)
            cpu_b = {"value": tok_s, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample}

    if rank == 0:
        setup = dict(cache_fill_s=round(t_fill, 1), weight_bytes=stage.weight_bytes(),
                     cache_bytes_per_layer=kd.layer_step_bytes(cfg, L), table_precision=stage.layers[0].cache.precision,
                     sp_exchange=sp_exchange)
        line = dict(base, value=value, ms_per_step=ms_step, config=config, setup=setup, clocks=clocks,
                    e2e={"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": 8,
                         "d2h_bytes_per_step": cfg.vocab * 2},
                    gpu_launches=int(launches_per_step * args.steps), roofline=roof, cpu_baseline=cpu_b)
        print(json.dumps(line), flush=True)
    if world > 1:
        # tear-down: graphs that captured NCCL kernels must die before the communicator; a hung destroy must not hold
        # the job (the result line is already out), so leave through os._exit after a final barrier
        sys.stdout.flush()
        del gs
        torch.cuda.synchronize()
        dist.barrier()
        os._exit(0)
    return 0


if __name__ == "__main__":
    sys.exit(main())
