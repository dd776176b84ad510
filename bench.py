#!/usr/bin/env python
"""Benchmark of the LineTR hot path: image-pairs/s of (encode side 0 + encode side 1 + match) on
synthetic 640x480 frames, weak scaling over 1..8 GPUs (pairs are independent; one all-gather of
per-pair match counts).

    python bench.py [--gpus N --steps K --warmup W] [--workload cfg1|cfg2|cfg3|cfg4]   # this repo's CUDA path
    python bench.py --impl reference [...]                                             # CPU baseline (oracle port)
    python bench.py [...] --dump-outputs DIR      # also write what the last timed step returned, DIR/<name>.npy


Workloads (BASELINE.json `configs`; per GPU, weak scaling):
    cfg1  64 pairs x 128 lines x 21 tokens x d256        (the headline configuration, default)
    cfg2  64 pairs x 256 lines x 32 tokens                (512 pairs over 8 GPUs)
    cfg3  64 pairs, ragged 32..512 lines/image, 64 token slots, 5..64 real tokens/line (256 pairs over 4 GPUs)
    cfg4  matcher only: 64 pairs x (1024 x 1024) x d256

Prints ONE JSON line: `value` = pairs/s with inputs resident in
HBM, `e2e` = the same through pinned-host buffers (H2D of every input tensor and D2H of the match
indices inside the timed region), `roofline` for the dominant kernel class (a second pass of the same
K steps with a CUDA-event pair around every launch on the launching stream; separate so that the
events do not serialise the kernels of the timed pass), `cpu_baseline` (oracle port on the host
cores: median of >= 10 single-pair calls after 3 warm-ups, in a subprocess with the BLAS/OpenMP
thread count pinned; one leg per thread setting, the best one is the baseline).

Multi-GPU (torchrun): the per-pair match counts of all ranks reach every rank each step - by default stored by the matcher's
tail kernel into every rank's symmetric buffer over NVLink (`LTR_BENCH_GATHER=p2p`), or `LTR_BENCH_GATHER=nccl` (all-gather);
`off` and `LTR_BENCH_KEEP=n` (exchanges left in flight across a step boundary, default 1) exist for diagnosis.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "image-pairs/s (line-descriptor forward x2 + mutual-NN match)"
UNIT = "pairs/s"
DTYPE = "f32 io / split-bf16 x3 tensor-core products, fp32 accumulate"
NCU_SUMMARY = os.path.join(ROOT, "profiles", "r2_ncu_summary.json")

WORKLOADS = {
    "cfg1": dict(pairs=64, lines=128, tokens=21, desc="cfg1: {P} pairs/GPU x 128 lines x 21 tokens x d256, 1 descriptive + 7 signature layers"),
    "cfg2": dict(pairs=64, lines=256, tokens=32, desc="cfg2: {P} pairs/GPU x 256 lines x 32 tokens x d256"),
    "cfg3": dict(pairs=64, lines=None, tokens=64, desc="cfg3: {P} pairs/GPU, ragged 32..512 lines/image, 64 token slots (5..64 real), d256"),
    "cfg4": dict(pairs=64, lines=1024, tokens=0, desc="cfg4: matcher only, {P} pairs/GPU x 1024 x 1024 lines x d256"),
    "tiny": dict(pairs=4, lines=16, tokens=5, desc="tiny: {P} pairs/GPU x 16 lines x 5 tokens (contract tests only)"),
}


def env_int(name, default):
    return int(os.environ.get(name, default))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch and kernel class, parsed from the committed
    `ncu --set full` summary of the FINAL kernels (tools/ncu_summary.py writes it); {} until one exists."""
    if os.path.exists(NCU_SUMMARY):
        with open(NCU_SUMMARY) as f:
            return json.load(f).get("traffic_bytes_per_launch", {})
    return {}


# ---------------------------------------------------------------- algorithmic work (SURVEY §8d)
def flops_per_image(L, T, n_sig=7):
    """Useful FLOPs (2*MAC) of one image under reference semantics (CLS row of the last layer)."""
    N = T + 1
    f_wpe = 217280 * L * T
    f_lpe = 217408 * L
    f_desc_cls = 4096 * L * N + 1310720 * L
    f_sig = (1310720 * L + 1024 * L * L) * n_sig
    f_fin = 131072 * L
    return f_wpe + f_lpe + f_desc_cls + f_sig + f_fin


def gemm_flops_per_image(L, T, n_sig=7):
    """Useful FLOPs the `linear` kernel class (gemm_img_kernel launches) is responsible for, one
    image: line stage (per-head V projection, fc, FFN, wide line-positional layers), signature
    layers (qkv, MLP with the merge projection folded in, MLP out) and final_proj.  The 3x
    split-bf16 products are NOT counted."""
    line = 2 * (4 * 256 * 64 + 256 * 256 + 2 * 256 * 1024 + 128 * 256 + 256 * 256) * L
    sig = 2 * (256 * 768 + 512 * 512 + 512 * 256) * L * n_sig
    fin = 2 * 256 * 256 * L
    return line + sig + fin


def token_flops_per_image(L, T):
    """Useful FLOPs of token_fused_kernel: narrow MLP 3-32-64, 64-128-256-256 on tensor cores, CLS pooling."""
    return (2 * (3 * 32 + 32 * 64 + 64 * 128 + 128 * 256 + 256 * 256) + 4096) * L * T


def bytes_per_image(L, T):
    return 4 * (256 * L * T + 2 * L * T + L * T + L * (T + 1) + 4 * L + L + 2 * L) + 4 * 256 * L


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.004)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------- synthetic workloads
def load_weights():
    """The shipped LineTR checkpoint when a copy travelled with the repo (SURVEY §8d), else seeded
    random-init weights of the same architecture (perf-neutral: same shapes, same kernels)."""
    from linetr_b200 import synthetic as syn
    p = os.path.join(ROOT, "linetr_b200", "weights", "LineTR_weight.pth")
    if os.path.exists(p):
        import torch
        return {k: v.numpy() for k, v in torch.load(p, map_location="cpu").items()}, "shipped LineTR_weight.pth"
    return syn.make_state_dict(0, 1), "random-init weights (seeded)"


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes {name: device tensor} as out_dir/<name>.npy: floating outputs as float32, integer ones as float64
    (exact).  Beyond DUMP_BUDGET_BYTES in all, every array is cut to the same fixed, seeded sample of its
    elements, whose flat indices go to <name>_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.detach().cpu().numpy().reshape(-1) for k, v in arrays.items()}
    host = {k: v.astype(np.float32 if v.dtype.kind == "f" else np.float64) for k, v in host.items()}
    frac = None
    if sum(v.nbytes for v in host.values()) > DUMP_BUDGET_BYTES:
        # a sampled element costs its value plus its float64 index; 4 KB per file for the two .npy headers
        cost = sum(v.size * (v.itemsize + 8) for v in host.values())
        frac = (DUMP_BUDGET_BYTES - 2 * 4096 * len(host)) / cost
    for k, v in host.items():
        if frac is not None:
            n = int(v.size * frac)
            idx = np.sort(np.random.Generator(np.random.PCG64(0)).choice(v.size, size=n, replace=False))
            np.save(os.path.join(out_dir, f"{k}_index.npy"), idx.astype(np.float64))
            v = v[idx]
        np.save(os.path.join(out_dir, f"{k}.npy"), v)


def cfg3_sizes(seed, n):
    rng = np.random.Generator(np.random.PCG64(seed))
    return [int(x) for x in rng.integers(32, 513, size=n)]


def make_pairs(workload, seed0, n):
    """-> list of (side0 dict, side1 dict) tokenizer-layout inputs (cfg1..3) or (d0 [256,n], d1 [256,n]) (cfg4)."""
    from linetr_b200 import synthetic as syn
    w = WORKLOADS[workload]
    if workload == "cfg4":
        return [syn.make_descriptor_pair(seed0 + i, 1024, 1024)[:2] for i in range(n)]
    if workload == "cfg3":
        Ls = cfg3_sizes(seed0, n)
        return [syn.make_pair_inputs(seed0 + i, Ls[i], 64, n_real_tokens=(5, 64))[:2] for i in range(n)]
    return [syn.make_pair_inputs(seed0 + i, w["lines"], w["tokens"])[:2] for i in range(n)]


# ---------------------------------------------------------------- CPU arm (oracle port), run in a subprocess
def cpu_worker(args):
    """Times single-pair calls of the CPU port (B = 1 per call, as Matching.forward runs the reference,
    models/matching.py:41,59,77-81) with the thread count this process was started with."""
    import torch
    torch.set_num_threads(args.threads)
    torch.set_grad_enabled(False)
    from oracle import linetr_oracle as orc
    from oracle import linetr_oracle_torch as port
    n_pairs = min(args.n + args.warm, 4) if args.workload != "cfg3" else min(args.n, 10)
    pairs = make_pairs(args.workload, 900, n_pairs)
    if args.workload == "cfg4":
        fn = lambda p: orc.nn_matcher(p[0], p[1], 0.8, True)
    else:
        sd = port.prepare(load_weights()[0])
        fn = lambda p: port.match_pair(sd, p[0], p[1])
    for i in range(args.warm):
        fn(pairs[i % len(pairs)])
    times = []
    for i in range(args.n):
        t0 = time.perf_counter()
        fn(pairs[i % len(pairs)])
        times.append(time.perf_counter() - t0)
    print(json.dumps({"times_s": times, "threads": args.threads, "torch_threads": torch.get_num_threads()}))


def decisive_rows(dist, thr, margin=4e-3):
    """Rows of a key-line distance matrix [K0,K1] whose match decision does not hinge on differences
    below `margin` (SURVEY 7 "hard parts": descriptors agree to 1e-3, so a top-2 gap, a threshold
    distance or the chosen column's own top-2 gap below ~4e-3 may legitimately flip)."""
    d = np.clip(np.asarray(dist, dtype=np.float64), 0.0, None)
    K0, K1 = d.shape
    if K0 == 0 or K1 == 0:
        return np.ones(K0, dtype=bool)
    srt = np.sort(d, axis=1)
    row_gap = srt[:, 1] - srt[:, 0] if K1 > 1 else np.full(K0, np.inf)
    idx = d.argmin(axis=1)
    csrt = np.sort(d, axis=0)
    col_gap = (csrt[1] - csrt[0]) if K0 > 1 else np.full(K1, np.inf)
    return (row_gap > margin) & (np.abs(srt[:, 0] - thr) > margin) & (col_gap[idx] > margin)


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_cpu_leg(workload, threads, n, warm):
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        env[k] = str(threads)
    env["CUDA_VISIBLE_DEVICES"] = ""
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    cmd = [sys.executable, os.path.abspath(__file__), "--cpu-worker", "--workload", workload, "--threads", str(threads),
           "--n", str(n), "--warm", str(warm)]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    if out.returncode != 0:
        raise RuntimeError(f"cpu worker failed: {out.stderr[-400:]}")
    r = json.loads(out.stdout.strip().splitlines()[-1])
    t = np.asarray(r["times_s"])
    ragged = workload == "cfg3"
    per_pair = float(t.mean()) if ragged else float(np.median(t))
    return {"threads": threads, "pairs_per_s": 1.0 / per_pair, "s_per_pair_median": float(np.median(t)),
            "s_per_pair_min": float(t.min()), "s_per_pair_max": float(t.max()), "n": int(len(t)), "warmup": warm,
            "stat": "mean over the ragged sample" if ragged else "median"}


def cpu_reference(workload, n=10, warm=3, quick=False):
    """All thread legs; the best one is the baseline ("all the host threads it can use" = the setting
    that makes the reference fastest; more threads than that slow torch-CPU/BLAS down on this path)."""
    ncpu = os.cpu_count() or 1
    # 1 / 8 / 16 / 32 threads: on the 128-thread GPU hosts the torch-OMP + BLAS pools of this B=1 path peak at
    # 8-16 threads and collapse beyond (measured there: 27 pairs/s at 8 threads, 0.03 pairs/s at 128), so
    # larger settings only burn minutes
    legs_t = sorted({1, min(8, ncpu), min(16, ncpu), min(32, ncpu)})
    if quick:
        legs_t = sorted({1, min(8, ncpu)})
    legs = [run_cpu_leg(workload, t, n, warm) for t in legs_t]
    best = max(legs, key=lambda l: l["pairs_per_s"])
    return best, legs


def cpu_baseline_obj(workload, best, legs, note=""):
    w = WORKLOADS[workload]
    what = "nn_matcher 1024x1024" if workload == "cfg4" else f"{w['lines'] or 'ragged 32..512'} lines x {w['tokens']} tokens"
    return {"value": best["pairs_per_s"], "unit": UNIT, "cores": best["threads"], "kind": "port",
            "host_cpus": os.cpu_count(), "cpu_model": cpu_model(),
            "sample": f"{best['stat']} of {best['n']} single-pair calls ({what}; B=1 per call as Matching.forward) after "
                      f"{best['warmup']} warm-ups, subprocess with OMP/MKL/OPENBLAS_NUM_THREADS={best['threads']}; "
                      "torch-CPU functional port of the reference (same aten ops)" + note,
            "legs": legs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg1", choices=sorted(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=0, help="image pairs per GPU per step (0 = the workload's own)")
    ap.add_argument("--e2e-chunks", type=int, default=4, help="pair groups whose H2D copy overlaps compute in the e2e leg")
    ap.add_argument("--profile-only", action="store_true", help="resident steps only (for runs under ncu)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank r > 0: <name>_rank<r>.npy)")
    ap.add_argument("--cpu-worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--threads", type=int, default=1, help=argparse.SUPPRESS)
    ap.add_argument("--n", type=int, default=10, help=argparse.SUPPRESS)
    ap.add_argument("--warm", type=int, default=3, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.cpu_worker:
        return cpu_worker(args)
    rank, world = env_int("RANK", 0), env_int("WORLD_SIZE", 1)
    local_rank = env_int("LOCAL_RANK", 0)
    wl = args.workload
    W = WORKLOADS[wl]
    P, L, T = args.pairs or W["pairs"], W["lines"], W["tokens"]
    config = {"workload": W["desc"].format(P=P), "name": wl, "pairs_per_gpu": P, "lines": L, "tokens": T,
              "sharding": f"pairs over {world} ranks"}

    if args.impl == "reference":
        if rank != 0:
            return
        # one step = one pair (B = 1 per call, as Matching.forward drives the reference); every thread setting gets the
        # full W warm-ups + K timed steps, the best leg is the value - the same rule as the cpu_baseline leg of the main
        # arm, so the two agree on one box
        leg, legs = cpu_reference(wl, n=max(args.steps, 1), warm=max(args.warmup, 1))
        value = leg["pairs_per_s"]
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": 1e3 * leg["s_per_pair_median"], "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded inputs); " + load_weights()[1],
               "config": config, "impl": "reference",
               "cpu_baseline": cpu_baseline_obj(wl, leg, legs, "; one step = one pair"),
               "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out))
        return

    import torch
    import torch.distributed as dist
    from linetr_b200 import LineBatch, LineTransformer, PairEngine, _native, _ops
    from linetr_b200.engine import PeerCounts, gather_counts

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    sd, wnote = load_weights()
    model = LineTransformer({"mode": "train", "max_tokens": max(T, 1)})
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    model = model.eval().to(dev)
    eng = PairEngine(model, dev)

    pairs = make_pairs(wl, 10_000 * (rank + 1), P)
    if wl == "cfg4":
        host0 = torch.from_numpy(np.concatenate([np.ascontiguousarray(a.T) for a, _ in pairs], 0)).pin_memory()
        host1 = torch.from_numpy(np.concatenate([np.ascontiguousarray(b.T) for _, b in pairs], 0)).pin_memory()
        res0, res1 = host0.to(dev), host1.to(dev)
        in_bytes = host0.numel() * 4 + host1.numel() * 4
        n_out = P * 1024
        Ls0 = Ls1 = [1024] * P
    else:
        # one packed batch: images [0, P) = side 0, [P, 2P) = side 1 (one encode launch sequence per step)
        host = LineBatch.from_images([a for a, _ in pairs] + [b for _, b in pairs]).pin()
        resident = host.to(dev)
        in_bytes = host.nbytes()
        Ls0 = [int(a["desc_sublines"].shape[1]) for a, _ in pairs]
        Ls1 = [int(b["desc_sublines"].shape[1]) for _, b in pairs]
        n_out = sum(Ls0)
    config["l2_policy"] = f"inputs {in_bytes / 1e6:.0f} MB per step > 126 MB L2"
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # The path's one collective (every rank learns all per-pair match counts).  Default: fused into the matcher's
    # tail kernel - its last block stores the counts into every rank's symmetric buffer over NVLink (multimem.st
    # / peer stores), no NCCL kernel competes with the persistent CTAs for an SM slot.  LTR_BENCH_GATHER=nccl:
    # ncclAllGather on NCCL's stream (the round-1 path).
    gather_mode = os.environ.get("LTR_BENCH_GATHER", "p2p") if world > 1 else "none"   # "off": diagnosis, no exchange at all
    peer = None
    if gather_mode == "p2p":
        try:
            peer = PeerCounts(P)
            gather_mode = "p2p-multimem" if peer.multicast else "p2p-stores"
        except Exception as e:   # symmetric memory unavailable: say so and use NCCL
            gather_mode = f"nccl (PeerCounts unavailable: {type(e).__name__})"
    config["count_gather"] = gather_mode
    pending = []   # all-gathers in flight: the gather of step i overlaps the kernels of step i+1
    gathered = {}

    KEEP = int(os.environ.get("LTR_BENCH_KEEP", "0"))   # diagnosis: gathers left in flight across a step boundary

    def drain(keep=0):
        while len(pending) > keep:
            h = pending.pop(0)[1]
            gathered["last"] = h.result() if peer is not None else h.wait()

    def run_resident(gather=None):
        """-> the arrays the caller of the path receives (on the device)."""
        if wl == "cfg4":
            out = _ops.match_descriptors(res0, res1, _native.LAYOUT_ROWS, P, 0.8, True, n0=1024, n1=1024, want_dist=False,
                                         gather=gather)
            return {k: out[k] for k in ("matches0", "scores0", "nn1", "counts")}
        res = eng.match_packed(resident, P, 0.8, gather=gather)
        return {"matches0": res.matches0, "scores0": res.scores0, "counts": res.counts,
                "offsets0": torch.from_numpy(res.offsets0)}

    def step_resident():
        if peer is not None:
            out = run_resident(peer.publish())
            # counts of step i-2: one exchange stays in flight across the step boundary.  A host that waits for the
            # previous step's counts (and the peers' flags) before it enqueues the next step lets the launch queue run dry
            # whenever the ranks drift into ping-pong - the same box measured 0.99 and 1.41 ms per step that way.  With
            # LTR_GATHER_SLOTS = 8 a peer can only overwrite a slot 8 steps later, when this rank has long read it.
            drain(max(KEEP, 1))
            pending.append((None, peer.collect_async())) # copy-engine D2H of this step's slot behind this step's kernels
            return out
        out = run_resident()
        if world > 1 and gather_mode != "off":
            # NCCL path: one all-gather stays in flight across the step boundary - its kernel has to find an SM between
            # persistent CTAs that follow each other without a gap (PDL), and a host that waits for it every step lets
            # the launch queue run dry (measured 1.41 ms per step against 1.05 ms)
            drain(max(KEEP, 1))
            pending.append(gather_counts(out["counts"], P * world, async_op=True))
        return out

    out_host = {"m": torch.empty(n_out, dtype=torch.int32).pin_memory(), "c": torch.empty(P, dtype=torch.int32).pin_memory()}

    def step_e2e():
        if wl == "cfg4":
            a, b = host0.to(dev, non_blocking=True), host1.to(dev, non_blocking=True)
            out = _ops.match_descriptors(a, b, _native.LAYOUT_ROWS, P, 0.8, True, n0=1024, n1=1024, want_dist=False)
            m0, cnt = out["matches0"], out["counts"]
        else:
            m0, cnt, _ = eng.match_packed_host(host, P, 0.8, n_chunks=args.e2e_chunks)
        out_host["m"].copy_(m0, non_blocking=True)
        out_host["c"].copy_(cnt, non_blocking=True)
        if world > 1:
            gather_counts(cnt, P * world)
        torch.cuda.current_stream().synchronize()   # the caller reads the result on the host

    for _ in range(args.warmup):
        step_resident()
    drain()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- timed region: K steps, inputs resident in HBM, CUDA events on the launching stream ----
    _native.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        timed_out = step_resident()
    drain()            # the last step's all-gather is inside the timed region
    e1.record()
    barrier()
    launches = _native.launch_count()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.result()
    # ---- the same K steps again with a CUDA-event pair around EVERY kernel launch (per-class device
    #      time for the roofline).  Kept out of the region above because an event record between two
    #      kernels serialises them and would switch off the programmatic dependent launch overlap. ----
    _native.profile_begin()
    for _ in range(args.steps):
        last = step_resident()
    drain()
    barrier()
    prof = _native.profile_end()
    m_last, c_last = last["matches0"], last["counts"]
    if args.dump_outputs:
        sfx = f"_rank{rank}" if rank else ""
        dump_outputs(args.dump_outputs, {k + sfx: v for k, v in timed_out.items()})

    if args.profile_only:
        return
    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0

    t = torch.tensor([ms_total, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms = float(t[0]), float(t[1])
    if rank == 0:
        # ---- output sanity: the matches of pair 0 of the timed batch against the CPU port (a silent kernel
        #      regression must not print a throughput) ----
        from oracle import linetr_oracle as orc
        from oracle import linetr_oracle_torch as port
        got0 = m_last[:Ls0[0]].cpu().numpy()
        if wl == "cfg4":
            mat0, dk0 = orc.nn_matcher(pairs[0][0], pairs[0][1], 0.8, True)
        else:
            with torch.no_grad():
                mat0, dk0 = port.match_pair(port.prepare(sd), pairs[0][0], pairs[0][1])[:2]
        want0 = orc.match_indices(mat0)
        dec = decisive_rows(dk0[0], 0.8)
        mism = int((got0 != want0)[dec].sum())
        check = {"pair0_indices_equal_cpu_port": mism == 0, "mismatches_on_decisive_rows": mism,
                 "rows": int(len(want0)), "decisive_rows": int(dec.sum()), "mismatches_all_rows": int((got0 != want0).sum()),
                 "matches_cpu_port": int((want0 >= 0).sum()), "matches_gpu": int(c_last[0])}
        assert mism == 0 and int(c_last[0]) == int((got0 >= 0).sum()), f"bench output check failed: {check}"

        peaks = load_peaks()
        traffic = load_traffic()
        ms_step = ms_total / args.steps
        value = P * world / (ms_step / 1e3)
        dom = max(prof.items(), key=lambda kv: kv[1][0]) if prof else ("none", (0.0, 0))
        dom_name, (dom_ms, dom_launches) = dom
        shares = {k: round(v[0] / max(sum(x[0] for x in prof.values()), 1e-9), 4) for k, v in prof.items()}
        sumL = sum(Ls0) + sum(Ls1)
        match_flops = sum(512 * a * b for a, b in zip(Ls0, Ls1))
        if wl == "cfg4":
            class_flops = {"match_tc": match_flops}
            useful_flops_step = match_flops
            alg_bytes_step = in_bytes + 8 * n_out
        else:
            class_flops = {"linear": sum(gemm_flops_per_image(l, T) for l in Ls0 + Ls1),
                           "token_fused": sum(token_flops_per_image(l, T) for l in Ls0 + Ls1),
                           "sig_attention": sum(7 * 1024 * l * l for l in Ls0 + Ls1),
                           "match_tc": match_flops}
            useful_flops_step = sum(flops_per_image(l, T) for l in Ls0 + Ls1) + match_flops
            alg_bytes_step = sum(bytes_per_image(l, T) for l in Ls0 + Ls1) + 8 * n_out
        class_kernel = {"linear": "gemm_img_kernel (tcgen05, split-bf16 x3, TMA-fed tile images)",
                        "token_fused": "token_fused_kernel (tcgen05 + CUDA-core pooling)",
                        "sig_attention": "sig_attention_tc_kernel (tcgen05)",
                        "match_tc": "match_tc_kernel (tcgen05 desc x desc^T both directions, row argmin in the epilogue)"}
        roof = None
        if dom_name in class_flops and dom_launches:
            per_launch_flops = class_flops[dom_name] * args.steps / dom_launches
            avg_ms = dom_ms / dom_launches
            ach = per_launch_flops / (avg_ms * 1e-3) / 1e12
            roof = {"bound": "tensor", "kernel": class_kernel[dom_name], "achieved": ach,
                    "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"],
                    "frac_of_sustained_peak": ach / peaks["bf16_tflops_sustained"],
                    "traffic": traffic.get(dom_name),
                    "peak_source": f"{peaks['source']} bf16 burst (MEASURED_PEAKS.json; the timed region is tens of ms at full clocks); "
                                   "useful FLOPs only",
                    "issued_over_useful_flops": 6.0 if dom_name == "match_tc" else 3.0,
                    "launches_per_step": dom_launches / args.steps, "avg_launch_ms": avg_ms,
                    "algorithmic_flops_per_launch": per_launch_flops}
        # secondary rooflines (same live per-class times)
        by_class = {}
        for name in ("sig_attention", "token_fused", "linear", "match_tc"):
            if name in prof and prof[name][1] and name in class_flops:
                ms_c, n_c = prof[name]
                tf = class_flops[name] * args.steps / (ms_c * 1e-3) / 1e12
                by_class[name] = {"kernel": class_kernel[name], "launches_per_step": n_c / args.steps,
                                  "avg_launch_ms": ms_c / n_c, "useful_tflops": tf,
                                  "frac_tensor_peak": tf / peaks["bf16_tflops"], "traffic": traffic.get(name)}
        if "token_fused" in by_class:
            tok_bytes = alg_bytes_step - 8 * n_out - 4 * 256 * sumL + 4 * 1024 * sumL   # inputs + z image (hi/lo bf16)
            gbs = tok_bytes * args.steps / (prof["token_fused"][0] * 1e-3) / 1e9
            by_class["token_fused"].update({"algorithmic_bytes_per_launch": tok_bytes * args.steps / prof["token_fused"][1],
                                            "hbm_gbs": gbs, "frac_hbm_peak": gbs / peaks["hbm_gbs"]})
        cpu = None
        if not args.no_cpu:
            best, legs = cpu_reference(wl, n=10, warm=3)
            cpu = cpu_baseline_obj(wl, best, legs)
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": DTYPE, "data": "synthetic (seeded inputs); " + wnote,
               "config": config, "clocks": clocks, "gpu_launches": int(launches),
               "e2e": {"value": P * world / (e2e_ms / 1e3 / args.steps), "unit": UNIT,
                       "h2d_bytes_per_step": in_bytes,
                       "d2h_bytes_per_step": out_host["m"].numel() * 4 + out_host["c"].numel() * 4},
               "roofline": roof,
               "useful_tflops": useful_flops_step / (ms_step * 1e-3) / 1e12,
               "hbm_gbs_algorithmic": alg_bytes_step / (ms_step * 1e-3) / 1e9,
               "kernel_time_shares": shares,
               "roofline_by_class": by_class,
               "output_check": check,
               "cpu_baseline": cpu}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
