#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): Chromoformer-clf default config, inference over 18,955
synthetic genes per GPU (configs[1]); genes/s, weak scaling over N GPUs with no collective.

    python bench.py [--gpus N --steps K --warmup W] [--mode infer|train] [--impl reference] [--dump-outputs DIR]

One JSON line on rank 0.  A "step" is one full sweep of the hot path over this rank's 18,955
genes.  `value` = genes of all ranks / max-over-ranks device time with inputs resident in HBM;
`e2e` = the same sweep through the public host API (pinned host buffers, H2D + D2H inside the
timed region).  `roofline` is for the dominant kernel (the batched dense projection of the
Regulation stack) timed alone with CUDA events; `cpu_baseline` / `--impl reference` time the
CPU oracle (a port of the reference's PyTorch-eager algorithm as written) on the host cores.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_GENES = 18955
KWS = ({"n_layers": 1, "n_heads": 2, "d_model": 128, "d_ff": 128},
       {"n_layers": 2, "n_heads": 2, "d_model": 128, "d_ff": 256},
       {"n_layers": 6, "n_heads": 8, "d_model": 256, "d_ff": 256})
BINS = (2000, 500, 100)


def ncu_traffic(kernel="reg_layer_fused_kernel"):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the committed export of the
    `ncu --set full` capture (profiles/r03_dense_ncu_metrics.json: the 18,955-gene launch of the final build, written by
    tools/ncu_extract.py; the 4096-gene capture of profiles/r02_ncu_metrics.json before it); None if absent."""
    path = os.path.join(ROOT, "profiles", "r03_dense_ncu_metrics.json")
    if not os.path.exists(path):
        path = os.path.join(ROOT, "profiles", "r02_ncu_metrics.json")
    try:
        d = json.load(open(path))[kernel]
        unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        rd = d["dram__bytes_read.sum"] * unit[d["dram__bytes_read.sum#unit"]]
        wr = d["dram__bytes_write.sum"] * unit[d["dram__bytes_write.sum#unit"]]
        return {"bytes": rd + wr, "read": rd, "write": wr, "source": "profiles/" + os.path.basename(path) + " (" + d.get("report", "?") + ")",
                "tensor_pipe_active_pct": max([v for k, v in d.items() if k.startswith("sm__pipe_tensor") and
                                               k.endswith("pct_of_peak_sustained_active") and isinstance(v, float)] or [None])}
    except (OSError, KeyError, ValueError):
        return None
REF_FLOPS_PER_GENE = 3862328832          # as-written forward, SURVEY §8d tier A


def executed_flops_per_gene(i_max=8, n_bins=(20, 80, 400), F=7, D=128):
    """FLOPs (2 x MAC) per gene of the formulation forward.cu actually executes (DESIGN.md §4)."""
    e, p, r = KWS
    S = i_max + 1
    mac = 0
    for n in n_bins:
        He, dme, dffe = e["n_heads"], D, e["d_ff"]
        sqa = lambda H, dm: dm * D + H * n * D + H * (2 * n * F + 2 * D * F) + H * n * D + dm * D
        mac += F * D + D * dme + sqa(He, dme) + dme * D + 2 * D * dffe                      # embedding, 1 row
        Hp, dmp, dffp = p["n_heads"], p["d_model"], p["d_ff"]
        mac += D * D + p["n_layers"] * i_max * (D * dmp + sqa(Hp, dmp) + dmp * D + 2 * D * dffp)
        Hr, dmr, dffr = r["n_heads"], r["d_model"], r["d_ff"]
        mac += r["n_layers"] * (S * (4 * dmr * D + dmr * D + 2 * D * dffr) + Hr * S * S * 32 * 2)
    mac += len(n_bins) * D * 128 + 128 * 2
    return 2 * mac


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  Samples are placed in time by nvidia-smi's
    own `timestamp` field (the reader thread can be starved of the GIL while the main thread launches kernels)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    @staticmethod
    def _epoch(stamp):
        # "2026/10/17 12:34:56.789" in local time
        try:
            head, _, ms = stamp.partition(".")
            return time.mktime(time.strptime(head, "%Y/%m/%d %H:%M:%S")) + (float("0." + ms) if ms else 0.0)
        except ValueError:
            return None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            ts = self._epoch(f[0]) if f else None
            self.rows.append((ts if ts is not None else time.time(), f[1:]))

    def window(self, t0, t1):
        """Samples taken in [t0, t1]."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.12)                      # let the reader thread drain what nvidia-smi has already written
        rows = [r for ts, r in list(self.rows) if t0 <= ts <= t1]
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


def make_model(cls, seed=123):
    return cls(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=seed)


# ------------------------------------------------------------------------------- CPU arm
REF_DIR = os.path.join(ROOT, "baseline", "_ref")        # `pip install --target baseline/_ref /root/reference` (DESIGN.md §2)


def _load_by_path(name, path):
    """Import one source file WITHOUT importing its package (the reference arm must not load this repo's package)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _reference_modules():
    """The UNMODIFIED reference package from baseline/_ref, on the CPU: `.cuda()` (hard-coded in net.py:52,129) is
    patched to the identity.  Returns (package, kind)."""
    import torch
    if not os.path.isdir(os.path.join(REF_DIR, "chromoformer")):
        return None, "port"
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self
    sys.path.insert(0, REF_DIR)
    for name in [m for m in sys.modules if m == "chromoformer" or m.startswith("chromoformer.")]:
        del sys.modules[name]
    import chromoformer
    assert os.path.abspath(chromoformer.__file__).startswith(REF_DIR), chromoformer.__file__
    return chromoformer, "reference"


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path (its PyTorch-eager modules, FP32, all
    host threads) on this arm's workload, in bounded samples: one step = one forward of 64 dense synthetic genes
    (train.py / run_demo.py batch sizes are 64 / 32).  Nothing of this repo's package or .so is loaded here."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    ref, kind = _reference_modules()
    syn = _load_by_path("chromo_synthetic_standalone", os.path.join(ROOT, "chromoformer_b200", "synthetic.py"))
    n_sample = args.ref_batch
    batch = syn.make_batch(n_sample, ragged=False, full_masks=True, seed=0)
    fargs = syn.forward_args(batch)
    if kind == "reference":
        model = ref.ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=123).eval()
        fwd = lambda: model(*fargs)
        what = "unmodified reference modules (baseline/_ref/chromoformer, PyTorch eager, CPU FP32)"
    else:       # reference package not staged: the oracle port of the same algorithm
        oracle = _load_by_path("chromo_oracle_standalone", os.path.join(ROOT, "oracle", "chromoformer_oracle.py"))
        sd = oracle.init_state_dict(regression=False, seed=123)
        fwd = lambda: oracle.chromoformer_forward(sd, *fargs)
        what = "oracle port of the as-written forward (oracle/chromoformer_oracle.py, torch CPU FP32)"
    with torch.no_grad():
        t0 = time.perf_counter()
        fwd()                                                     # first call also sizes the run
        first = time.perf_counter() - t0
        budget = 150.0                                            # the whole arm stays within a few minutes
        warmup = max(0, min(args.warmup, int(0.25 * budget / first)) - 1)
        steps = max(1, min(args.steps, int(0.75 * budget / first)))
        for _ in range(warmup):
            fwd()
        times = []
        for _ in range(steps):
            t0 = time.perf_counter()
            fwd()
            times.append(time.perf_counter() - t0)
    per = sum(times) / len(times)
    gps = n_sample / per
    extra = {}
    if not args.no_train and kind == "reference":
        extra["train"] = _reference_train_step(ref, syn, threads)
        extra["getitem"] = _reference_getitem(ref)
    line = {"impl": "reference", "metric": "genes/sec inference", "value": gps, "unit": "genes/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup + 1, "steps_requested": args.steps,
            "warmup_requested": args.warmup, "ms_per_step": per * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": workload_config(args),
            "cpu_baseline": {"value": gps, "unit": "genes/s", "cores": threads, "kind": kind,
                             "sample": f"{n_sample} dense synthetic genes per step x {steps} steps (median "
                                       f"{sorted(times)[len(times) // 2] * 1e3:.0f} ms): {what}",
                             "parallel_info": torch.__config__.parallel_info().split("\n")[1:3]},
            "e2e": {"value": gps, "unit": "genes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, **extra}
    print(json.dumps(line), flush=True)


def _reference_train_step(ref, syn, threads):
    """BASELINE.md §3: ChromoformerRegressor fwd + MSELoss + backward + torch.optim.AdamW.step, bsz 64, CPU FP32."""
    import torch
    model = ref.ChromoformerRegressor(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=123).train()
    opt = torch.optim.AdamW(model.parameters(), lr=3e-5)
    crit = torch.nn.MSELoss()
    b = syn.make_batch(64, ragged=False, full_masks=True, seed=100)
    fargs, target = syn.forward_args(b), b["labels_reg"].view(-1, 1)
    times = []
    for it in range(3):
        t0 = time.perf_counter()
        opt.zero_grad()
        loss = crit(model(*fargs), target)
        loss.backward()
        opt.step()
        times.append(time.perf_counter() - t0)
    per = min(times[1:])
    return {"metric": "train samples/sec", "value": 64 / per, "unit": "samples/s", "ms_per_step": per * 1e3, "cores": threads,
            "kind": "reference", "sample": "Chromoformer-reg bsz 64, 1 warm-up + best of 2 steps, unmodified reference + "
                                           "torch.optim.AdamW, CPU FP32"}


def _reference_getitem(ref):
    """BASELINE.md §3: the reference's ChromoformerDataset.__getitem__, one process, on the staged demo genes."""
    demo = os.path.join(REF_DIR, "demo")
    meta = os.path.join(demo, "demo_meta_head.csv")
    if not os.path.exists(meta):
        return None
    import pandas as pd
    genes = pd.read_csv(meta).gene_id.tolist()
    ds = ref.ChromoformerDataset(meta, os.path.join(demo, "demo_data"), genes, 7, 8, [2000, 500, 100], 40000, 40000)
    ds[0]
    t0 = time.perf_counter()
    for i in range(len(genes)):
        ds[i]
    per = (time.perf_counter() - t0) / len(genes)
    return {"metric": "ChromoformerDataset.__getitem__", "value": 1.0 / per, "unit": "genes/s/process", "ms_per_gene": per * 1e3,
            "kind": "reference", "sample": f"{len(genes)} staged demo genes, one process (data.py:115-212)"}


def cpu_baseline_subprocess(steps=3, warmup=1, train=True):
    """The b200 arm's `cpu_baseline`: the reference arm above in its OWN process (so that neither this repo's .so nor its
    `chromoformer` shim is anywhere near the timed reference code)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", str(warmup)]
    if not train:
        cmd.append("--no-train")
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env).stdout.strip().splitlines()
        return json.loads(out[-1])
    except Exception as e:                                        # noqa: BLE001
        return {"error": repr(e)}


def workload_config(args):
    return {"workload": "Chromoformer-clf default config (i_max=8, binsizes 2000/500/100, 7 marks) inference over "
                        "18,955 synthetic genes per GPU", "genes_per_gpu": N_GENES, "chunk": args.chunk, "e2e_chunk": args.e2e_chunk,
            "i_max": 8, "l2_policy": "inputs (2.5 GB/GPU) larger than L2; no flush needed",
            "precision": args.precision}


# ------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="timed sweeps of the headline region (`value`); the ragged and e2e figures derive their own "
                         "counts from it, and a headline region under 0.6 s is followed by a separate `sustained` one")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--mode", choices=["infer", "train"], default="infer")
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--chunk", type=int, default=N_GENES,
                    help="genes per launch chain of the device-resident sweep (default: the whole sweep; measured on one B200 "
                         "4096: 2.98, 6216: 3.07, 9478: 3.25, 18955: 3.38 M genes/s, tools/chunk_sweep.py)")
    ap.add_argument("--e2e-chunk", type=int, default=4096, help="genes per host->device copy / forward chunk of the e2e arm")
    ap.add_argument("--precision", choices=["fp32", "bf16"], default="bf16")
    ap.add_argument("--train-precision", choices=["fp32", "bf16"], default="bf16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--ref-batch", type=int, default=64, help="genes per step of the CPU reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the logits of the last timed sweep of the headline region (rank 0's genes) to "
                         "DIR/logits.npy in float32; the inputs and weights are seeded, so two builds run with the same "
                         "arguments compare array for array (not with --impl reference)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args)
        return

    # keep stdout clean for the ONE JSON line: NCCL prints its version banner to stdout at init
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import torch.distributed as dist
    from chromoformer_b200 import ChromoformerClassifier, ChromoformerRegressor, _lib, synthetic
    from chromoformer_b200.engine import InferenceEngine, batch_nbytes, pack_wire, pin_batch, wire_nbytes
    from chromoformer_b200.parallel import bind_to_gpu_numa
    from chromoformer_b200.trainer import TrainStep

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_note = bind_to_gpu_numa(local)          # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    peaks = load_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps

    # ---------------- inference: device-resident sweep ----------------------------------
    model = make_model(ChromoformerClassifier).cuda().eval()
    model.precision = args.precision
    host = synthetic.make_batch(N_GENES, ragged=False, seed=rank)        # dense: k = 8, full-length pCREs
    eng = InferenceEngine(model, chunk=args.chunk)
    resident = eng.to_device(host)
    out = torch.empty(N_GENES, 2, device=dev)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                                                     # (nvidia-smi needs a moment to come up)
    eng.predict_device(resident, out)                                       # first touch / workspace allocation
    torch.cuda.synchronize()
    lib.chromo_launch_counter(1)
    eng.predict_device(resident, out)
    launches_per_step = int(lib.chromo_launch_counter(1))
    t0 = time.time()
    ms = timed(lambda: eng.predict_device(resident, out), args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "logits.npy"), out.cpu().numpy())
    # `value` is EXACTLY --steps sweeps (the driver's contract); a short region (20 steps = 0.13 s) is followed by a second,
    # >= 0.6 s region of the same step so that the clock samples and a sustained figure exist regardless of --steps
    sustained = None
    if ms * args.steps < 600.0:
        n2 = int(600.0 / ms) + 1
        ms2 = timed(lambda: eng.predict_device(resident, out), n2, 0)
        sustained = {"steps": n2, "ms_per_step": ms2, "value": world * N_GENES / (ms2 * 1e-3), "unit": "genes/s"}
    t1 = time.time()
    clocks = None
    if rank == 0:
        clocks = sampler.window(t0, t1)
        if not clocks["samples"]:
            # the timed region is shorter than nvidia-smi's 100 ms sampling period: keep the same step running (untimed)
            # for 0.6 s right behind it and sample that
            te = time.time()
            while time.time() - te < 0.6:
                eng.predict_device(resident, out)
                torch.cuda.synchronize()
            clocks = sampler.window(te, time.time())
            clocks["note"] = ("no nvidia-smi sample fell inside the timed region (%.0f ms); sampled over 0.6 s of the same "
                              "step run directly behind it" % ((t1 - t0) * 1e3))
        sampler.stop()
    genes_per_s = world * N_GENES / (ms * 1e-3)

    # ---------------- configs[3]: ragged genes (0..8 pCREs, demo-like lengths), same sweep size ----------------
    del resident
    rag_host = synthetic.make_batch(N_GENES, ragged=True, seed=1000 + rank)
    rag = eng.to_device(rag_host)
    rag_steps = max(5, args.steps // 4)
    ms_rag = timed(lambda: eng.predict_device(rag, out), rag_steps, 3)
    lib.chromo_launch_counter(1)
    eng.predict_device(rag, out)
    rag_launches = int(lib.chromo_launch_counter(1))
    # the same genes with the plan switched off (every slot, every bin computed), and the dense batch WITH the plan
    # (what a caller pays who does not pass the CHROMO_F_DENSE hint the engine derives on the host)
    rag["dense"] = True
    ms_rag_off = timed(lambda: eng.predict_device(rag, out), rag_steps, 3)
    del rag, rag_host
    dense_dev = eng.to_device(host)
    dense_dev["dense"] = False
    ms_dense_plan = timed(lambda: eng.predict_device(dense_dev, out), rag_steps, 3)
    del dense_dev
    ragged = {"what": "same sweep over ragged genes (pCRE count ~ demo histogram, valid 100-bp bins mean ~63 of 400): the "
                      "ragged plan (csrc/ragged.cu) drops dummy pCRE slots and padded bins, exactly",
              "value": world * N_GENES / (ms_rag * 1e-3), "unit": "genes/s", "ms_per_step": ms_rag,
              "gpu_launches_per_step": rag_launches,
              "without_plan": {"value": world * N_GENES / (ms_rag_off * 1e-3), "ms_per_step": ms_rag_off},
              "vs_dense": ms / ms_rag,
              "dense_batch_with_plan": {"value": world * N_GENES / (ms_dense_plan * 1e-3), "ms_per_step": ms_dense_plan,
                                        "what": "the headline batch without the CHROMO_F_DENSE hint"}}
    resident = eng.to_device(host)

    # ---------------- inference: end-to-end through the host API ---------------------------
    # headline `e2e`: the FP16 / span wire format (engine.pack_wire -> predict_wire): pinned host buffers, H2D of every
    # chunk + chromo_unpack_wire + forward + D2H of the logits, all inside the timed region.  Variants for context:
    # the FP32 compact layout (round 1's e2e), the reference's own collation (FP32 + n x n masks, 1.63 MB per gene, on a
    # 1024-gene sample) and raw .npy files through GeneBatcher (the staged demo genes).
    # headline wire: zero-suppressed FP16 features (occupancy bitmap + non-zero values; ln(mean + 1) is exactly 0 where no
    # read fell - 37 % of the bins of the demo set, which the synthetic feature law reproduces) + spans; lossless
    wire = pack_wire(host, sparse=True)
    h2d = wire_nbytes(wire)
    zero_frac = float(sum((t == 0).sum().item() for k in ("promoter_feats", "pcre_feats") for t in host[k].values())) / \
        float(sum(t.numel() for k in ("promoter_feats", "pcre_feats") for t in host[k].values()))
    e2e_steps = max(2, args.steps // 2)
    eng_res = eng
    eng = InferenceEngine(model, chunk=args.e2e_chunk)      # chunks: the copy of chunk i+1 runs under the forward of chunk i
    ms_e2e = timed(lambda: eng.predict_wire(wire), e2e_steps, 3)
    e2e = {"value": world * N_GENES / (ms_e2e * 1e-3), "unit": "genes/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": N_GENES * 2 * 4, "ms_per_step": ms_e2e,
           "api": "InferenceEngine.predict_wire(pack_wire(batch, sparse=True))",
           "format": "zero-suppressed FP16 features (occupancy bitmap + non-zero values, lossless; chromo_unpack_sparse) + "
                     "(first valid bin, count) spans; FP32 features / masks rebuilt on the device",
           "feature_zero_fraction": zero_frac,
           "h2d_bytes_per_gene": h2d / N_GENES, "h2d_gbs": world * h2d / (ms_e2e * 1e-3) / 1e9,
           "bound": "PCIe host->device copy", "numa": numa_note, "variants": {}}
    del wire
    wire = pack_wire(host)
    ms_v = timed(lambda: eng.predict_wire(wire), max(2, e2e_steps // 2), 2)
    e2e["variants"]["fp16_spans"] = {"value": world * N_GENES / (ms_v * 1e-3), "unit": "genes/s", "ms_per_step": ms_v,
                                     "h2d_bytes_per_gene": wire_nbytes(wire) / N_GENES,
                                     "h2d_gbs": world * wire_nbytes(wire) / (ms_v * 1e-3) / 1e9,
                                     "what": "every FP16 feature value + spans (no zero suppression)"}
    del wire
    pinned = pin_batch(host)
    ms_v = timed(lambda: eng.predict_host(pinned), max(2, e2e_steps // 2), 2)
    e2e["variants"]["fp32_compact"] = {"value": world * N_GENES / (ms_v * 1e-3), "unit": "genes/s", "h2d_bytes_per_gene": batch_nbytes(pinned) / N_GENES,
                                       "what": "FP32 features + centre-row masks (round 1's e2e)"}
    del pinned
    n_full = 1024
    full = pin_batch(synthetic.expand_full_masks(synthetic.slice_batch(host, 0, n_full)))
    eng_full = InferenceEngine(model, chunk=256)
    ms_v = timed(lambda: eng_full.predict_host(full), 3, 1)
    e2e["variants"]["reference_collated"] = {"value": world * n_full / (ms_v * 1e-3), "unit": "genes/s",
                                             "h2d_bytes_per_gene": batch_nbytes(full) / n_full,
                                             "what": "the reference DataLoader's own collation (FP32 + [B,8,1,n,n] boolean masks), "
                                                     f"{n_full}-gene sample in chunks of 256"}
    del full, eng_full
    # ragged genes (configs[3]) end to end: the compact wire ships only the valid bins of the live pCRE slots
    # (data.py:86-97,175-177 pads everything else with zeros), the forward runs under the ragged plan
    rag_host = synthetic.make_batch(N_GENES, ragged=True, seed=1000 + rank)
    for key, compact in (("ragged_fp16_spans", False), ("ragged_compact_wire", True)):
        rw = pack_wire(rag_host, compact=compact)
        ms_v = timed(lambda: eng.predict_wire(rw), max(2, e2e_steps // 2), 2)
        e2e["variants"][key] = {"value": world * N_GENES / (ms_v * 1e-3), "unit": "genes/s", "ms_per_step": ms_v,
                                "h2d_bytes_per_gene": wire_nbytes(rw) / N_GENES,
                                "h2d_gbs": world * wire_nbytes(rw) / (ms_v * 1e-3) / 1e9,
                                "what": "ragged genes (pCRE count ~ demo histogram, ~63 of 400 valid 100-bp bins), " +
                                        ("pCREs as their valid bins only (engine.pack_wire(compact=True) -> chromo_unpack_compact)" if compact
                                         else "every FP16 feature value + spans")}
        del rw
    del rag_host
    demo_dir = os.path.join(ROOT, "baseline", "_ref", "demo")
    if os.path.exists(os.path.join(demo_dir, "demo_meta_head.csv")) and rank == 0:
        import pandas as pd
        from chromoformer_b200.data import ChromoformerDataset, GeneBatcher
        meta = os.path.join(demo_dir, "demo_meta_head.csv")
        genes = pd.read_csv(meta).gene_id.tolist()
        ds = ChromoformerDataset(meta, os.path.join(demo_dir, "demo_data"), genes)
        gb = GeneBatcher(ds, device=dev, cache=False)

        def raw_npy():
            b = gb.batch(list(range(len(genes))))
            with torch.no_grad():
                return model.forward_batch(b).cpu()
        raw_npy()
        t0 = time.perf_counter()
        for _ in range(3):
            raw_npy()
        dt = (time.perf_counter() - t0) / 3
        e2e["variants"]["raw_npy_genebatcher"] = {"value": len(genes) / dt, "unit": "genes/s", "genes": len(genes),
                                                  "what": "np.load of the staged demo regions (page cache) -> pinned FP16 -> device binning "
                                                          "kernel -> forward -> host, one process, no DataLoader (reference __getitem__: "
                                                          "see cpu_baseline.getitem)"}

    # ---------------- dominant kernel alone ----------------------------------------------------
    # BF16: the fused Regulation layer (reg_layer_fused_kernel, 1/3 of the step); FP32: the batched projection GEMM.
    st = torch.cuda.current_stream().cuda_stream
    flags = _lib.F_BF16 if args.precision == "bf16" else 0
    Bk = min(args.chunk, N_GENES)
    T = Bk * 9
    if args.precision == "bf16":
        cfgk = _lib.Config.from_buffer_copy(model._cfg)
        xk = torch.randn(3, T, 128, device=dev)
        yk = torch.empty_like(xk)
        nws = _lib.check(lib.chromo_workspace_floats(ctypes.byref(cfgk), Bk, flags), "ws")
        wsk = torch.empty(nws, device=dev)
        imk = [resident["interaction_masks"][b][:Bk].contiguous() for b in BINS]
        imp = (ctypes.c_void_p * 3)(*[m.data_ptr() for m in imk])
        fqk = resident["interaction_freq"][:Bk].contiguous()
        state = {"flags": flags}

        n_lay = int(cfgk.reg_layers)

        def one_kernel():       # layer = -1: the whole Regulation transformer in one launch, as the forward runs it
            _lib.check(lib.chromo_regulation_layer(ctypes.byref(cfgk), model.flat_params.data_ptr(), -1, xk.data_ptr(),
                                                   yk.data_ptr(), T * 128, imp, fqk.data_ptr(), Bk, wsk.data_ptr(), nws,
                                                   state["flags"], st), "chromo_regulation_layer")
        one_kernel()                                   # packs the weight stream once
        state["flags"] = flags | _lib.F_PACKED
        ms_k = timed(one_kernel, 20, 5)
        flops_k = n_lay * 3.0 * T * 2 * (4 * 256 * 128 + 256 * 128 + 2 * 128 * 256 + 8 * 9 * 32 * 2)
        bytes_k = 2.0 * 3 * T * 128 * 4 + n_lay * 3 * 14 * 32768
        kname = (f"reg_layer_fused_kernel<9>: the {n_lay} Regulation layers in one launch, 3 resolutions x {T} tokens "
                 "(per layer: proj + tensor-pipe attention + out-proj/LN + FFN/LN; tcgen05 + TMA weight stream)")
        traffic = ncu_traffic()
        # second kernel: the fused single-query attention core at n = 400 (HBM-bound: 11.2 KB of features per region)
        nreg_s = Bk * 8
        g = torch.Generator(device="cpu").manual_seed(1)
        qk_s = torch.randn(nreg_s * 2, 128, device=dev) * 0.1
        x_s = resident["pcre_feats"][100][:Bk].reshape(nreg_s, 400, 7).contiguous()
        mk_s = torch.zeros(nreg_s, 400, dtype=torch.uint8, device=dev)
        win_s = torch.randn(128, 7, device=dev) * 0.1
        from chromoformer_b200.model import sinusoid_table
        pe_s = sinusoid_table(400, 128).to(dev)
        cb_s = torch.empty(nreg_s * 2, 128, device=dev)
        ws_s = torch.empty(64 * 400 + 1024 + 8192 * ((nreg_s + 63) // 64), device=dev)

        def one_sqa():
            _lib.check(lib.chromo_single_query_attention(nreg_s, 400, qk_s.data_ptr(), x_s.data_ptr(), mk_s.data_ptr(),
                                                         win_s.data_ptr(), pe_s.data_ptr(), 0.125, cb_s.data_ptr(),
                                                         ws_s.data_ptr(), ws_s.numel(), st), "chromo_single_query_attention")
        ms_s = timed(one_sqa, 20, 5)
        bytes_s = nreg_s * (400 * 7 * 4 + 400 + 2 * 128 * 4 * 2)
        sqa_line = {"kernel": "sqa_fused_kernel, n = 400 (scores + online softmax + both position-table GEMMs in TMEM)",
                    "bound": "hbm", "regions": nreg_s, "ms_per_launch": ms_s, "algorithmic_bytes": bytes_s,
                    "achieved": bytes_s / (ms_s * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": bytes_s / (ms_s * 1e-3) / 1e9 / peaks["hbm_gbs"],
                    "tflops": nreg_s * 2 * 2.0 * (2 * 128 * 400) / (ms_s * 1e-3) / 1e12}
    else:
        x = torch.randn(3, T, 128, device=dev)
        wgt = torch.randn(3, 1024, 128, device=dev)
        y = torch.empty(3, T, 1024, device=dev)

        def one_kernel():
            _lib.check(lib.chromo_linear(x.data_ptr(), wgt.data_ptr(), None, y.data_ptr(), T, 1024, 128, 0, 3,
                                         T * 128, 1024 * 128, 0, T * 1024, flags, st), "chromo_linear")
        ms_k = timed(one_kernel, 20, 5)
        flops_k = 2.0 * 3 * T * 1024 * 128
        bytes_k = 3.0 * T * (128 + 1024) * 4
        kname = f"gemm_simt_kernel<64,64> (FP32 CUDA cores) as launched for regulation.*.self_att.att (M={T}, N=1024, K=128, x3)"
        traffic = None
        sqa_line = None
    ach = flops_k / (ms_k * 1e-3) / 1e12
    fpg = executed_flops_per_gene()
    roofline = {"bound": "tensor", "kernel": kname, "achieved": ach, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": ach / peaks["bf16_tflops"], "traffic": traffic,
                "peak_source": peaks["source"] + " burst (kernel timed alone)", "ms_per_launch": ms_k,
                "algorithmic_flops_per_launch": flops_k, "algorithmic_bytes_per_launch": bytes_k,
                "hbm_frac": bytes_k / (ms_k * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "whole_forward": {"executed_flops_per_gene": fpg,
                                  "achieved_tflops": fpg * genes_per_s / world / 1e12,
                                  "reference_equivalent_tflops": REF_FLOPS_PER_GENE * genes_per_s / world / 1e12,
                                  "algorithmic_bytes_per_gene": 126000 + 4500 + 324 * 4,
                                  "achieved_gbs": (126000 + 4500 + 1296) * genes_per_s / world / 1e9,
                                  "hbm_peak_gbs": peaks["hbm_gbs"]}}

    # ---------------- input path kernel (data.py:68-113 on the device): HBM-bound byte work -------
    n_reg, L = 4096, 40000                                  # 2.29 GB of FP16 depth: larger than L2
    raw = (torch.rand(n_reg * 7 * L // 2, device=dev) * 3).to(torch.float16)
    raw = torch.cat([raw, raw])[: n_reg * 7 * L]
    table = np.zeros(n_reg, dtype=[("offset", "<i8"), ("length", "<i4"), ("start", "<i4"), ("width", "<i4"), ("flip", "<i4")])
    table["offset"] = np.arange(n_reg, dtype=np.int64) * 7 * L
    table["length"], table["width"], table["flip"] = L, L, np.arange(n_reg) % 2
    tab = torch.from_numpy(table.view(np.uint8).reshape(-1)).to(dev)
    feats = [torch.empty(n_reg, n, 7, device=dev) for n in (20, 80, 400)]
    spans = torch.empty(3, n_reg, 2, dtype=torch.int32, device=dev)
    ptrs = (ctypes.c_void_p * 3)(*[f.data_ptr() for f in feats])
    bins_c, nb_c = (ctypes.c_int32 * 3)(2000, 500, 100), (ctypes.c_int32 * 3)(20, 80, 400)

    def one_bin():
        _lib.check(lib.chromo_bin_regions(raw.data_ptr(), tab.data_ptr(), n_reg, 7, 3, bins_c, nb_c, ptrs,
                                          spans.data_ptr(), st), "chromo_bin_regions")
    ms_b = timed(one_bin, 10, 3)
    bytes_b = n_reg * 7 * L * 2 + n_reg * 500 * 7 * 4
    input_path = {"kernel": "bin_regions_fast_kernel", "bound": "hbm", "regions": n_reg, "bp_per_region": L,
                  "algorithmic_bytes": bytes_b, "ms_per_launch": ms_b, "achieved": bytes_b / (ms_b * 1e-3) / 1e9,
                  "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": bytes_b / (ms_b * 1e-3) / 1e9 / peaks["hbm_gbs"],
                  "regions_per_s": n_reg / (ms_b * 1e-3)}
    del raw, feats

    # ---------------- raw-depth path: FP16 depth in HBM -> binning kernel -> forward (no host work) ---------------
    # Two feature sets: the (HBM-bound) binning of batch i+1 runs on a side stream under the (tensor / latency-bound)
    # forward of batch i; pad masks come from the kernel's valid spans in one chromo_unpack_wire launch.
    Bq = 4096
    nreg = Bq * 9                                            # promoters first, then the 8 pCREs of every gene (40 kb each)
    blk = (torch.rand(nreg * 7 * L // 16, device=dev) * 3).to(torch.float16)        # (1.3 GB block, repeated: > L2)
    rawq = blk.repeat(16)[: nreg * 7 * L]
    del blk
    tq = np.zeros(nreg, dtype=table.dtype)
    tq["offset"] = np.arange(nreg, dtype=np.int64) * 7 * L
    tq["length"], tq["width"] = L, L
    tq["flip"][:Bq] = np.arange(Bq) % 2
    tabq = torch.from_numpy(tq.view(np.uint8).reshape(-1)).to(dev)
    NB = (20, 80, 400)
    fq = [[torch.empty(nreg, n, 7, device=dev) for n in NB] for _ in range(2)]
    sq = [torch.empty(3, nreg, 2, dtype=torch.int32, device=dev) for _ in range(2)]
    mq = [[torch.empty(nreg, n, dtype=torch.bool, device=dev) for n in NB] for _ in range(2)]
    imq = {b: resident["interaction_masks"][b][:Bq] for b in BINS}
    frq = resident["interaction_freq"][:Bq]
    side = torch.cuda.Stream(dev)
    fwd_s = torch.cuda.Stream(dev, priority=-1)              # the forward's CTAs go first whenever a binning block retires
    binned = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    arr = lambda ty, xs: (ty * len(xs))(*xs)

    def bin_set(k, stream):
        pq = arr(ctypes.c_void_p, [f.data_ptr() for f in fq[k]])
        _lib.check(lib.chromo_bin_regions(rawq.data_ptr(), tabq.data_ptr(), nreg, 7, 3, bins_c, nb_c, pq, sq[k].data_ptr(),
                                          stream.cuda_stream), "chromo_bin_regions")
        _lib.check(lib.chromo_unpack_wire(0, arr(ctypes.c_void_p, [0]), arr(ctypes.c_void_p, [0]), arr(ctypes.c_int64, [0]), 3,
                                          arr(ctypes.c_void_p, [sq[k][r].data_ptr() for r in range(3)]),
                                          arr(ctypes.c_void_p, [m.data_ptr() for m in mq[k]]),
                                          arr(ctypes.c_int32, [nreg] * 3), arr(ctypes.c_int32, list(NB)), stream.cuda_stream),
                   "chromo_unpack_wire")

    def forward_set(k):
        batch = {"promoter_feats": {}, "promoter_pad_masks": {}, "pcre_feats": {}, "pcre_pad_masks": {},
                 "interaction_masks": imq, "interaction_freq": frq}
        for r, (b, n) in enumerate(zip(BINS, NB)):
            batch["promoter_feats"][b] = fq[k][r][:Bq].view(Bq, 1, n, 7)
            batch["pcre_feats"][b] = fq[k][r][Bq:].view(Bq, 8, n, 7)
            batch["promoter_pad_masks"][b] = mq[k][r][:Bq].view(Bq, 1, n)
            batch["pcre_pad_masks"][b] = mq[k][r][Bq:].view(Bq, 8, n)
        with torch.no_grad():
            return model.forward_batch(batch, dense=True)            # (full-length regions: nothing is padded)

    state = {"cur": 0}
    main_s = torch.cuda.current_stream(dev)
    bin_set(0, main_s)
    binned[0].record(main_s)
    freed[1].record(main_s)

    def raw_step():
        k = state["cur"]
        side.wait_event(freed[1 - k])                        # the forward that read set 1-k is through
        with torch.cuda.stream(side):
            bin_set(1 - k, side)
            binned[1 - k].record(side)
        fwd_s.wait_stream(main_s)
        fwd_s.wait_event(binned[k])
        with torch.cuda.stream(fwd_s):
            res = forward_set(k)
            freed[k].record(fwd_s)
        main_s.wait_stream(fwd_s)
        state["cur"] = 1 - k
        return res
    ms_r = timed(raw_step, 6, 3)

    def raw_serial():
        bin_set(0, main_s)
        return forward_set(0)
    torch.cuda.synchronize()
    ms_rs = timed(raw_serial, 4, 2)
    raw_path = {"what": "raw FP16 depth resident in HBM -> chromo_bin_regions (+ masks from its spans) -> forward, 4096 dense "
                        "genes per step, the binning of batch i+1 on a side stream under the forward of batch i (forward on a high-priority stream)",
                "value": world * Bq / (ms_r * 1e-3), "unit": "genes/s", "ms_per_step": ms_r,
                "raw_bytes_per_gene": 9 * 7 * L * 2, "hbm_gbs": Bq * 9 * 7 * L * 2 / (ms_r * 1e-3) / 1e9,
                "one_stream": {"value": world * Bq / (ms_rs * 1e-3), "ms_per_step": ms_rs},
                "bound": "reading 5.04 MB of raw depth per gene: %.2f M genes/s at the measured HBM peak" % (peaks["hbm_gbs"] * 1e9 / (9 * 7 * L * 2) / 1e6)}
    del rawq, fq, mq, sq

    # ---------------- ensemble sweep (configs[4]): 44 checkpoints x this rank's share of (checkpoint, chunk) units ----
    sweep = None
    if not args.no_sweep:
        from chromoformer_b200.sweep import EnsembleSweep
        # (two chunks per checkpoint on several ranks: 88 units split evenly over 2, 4 and 8 ranks)
        es = EnsembleSweep(model, chunk=args.chunk if world == 1 else (N_GENES + 1) // 2)
        base = model.flat_params.detach().clone()
        gsw = torch.Generator(device=dev).manual_seed(1)
        for ck in range(44):                                  # 44 distinct random-init "checkpoints" (no weights offline)
            es.flats.append(base + 1e-3 * torch.randn(base.shape, generator=gsw, device=dev))
        units = None

        def sweep_step():
            nonlocal units
            units, _ = es.run(resident, rank=rank, world=world)
        ms_s = timed(sweep_step, 2, 1)
        evals = sum(g1 - g0 for (_, g0, g1) in units)
        model.flat_params.copy_(base)
        model.mark_parameters_changed()
        sweep = {"what": "44 checkpoints x 18,955 genes, (checkpoint, gene-chunk) units sharded over ranks, no collective",
                 "gene_evaluations_per_rank": evals, "ms": ms_s, "value": world * evals / (ms_s * 1e-3) if world == 1 else None,
                 "per_rank_value": evals / (ms_s * 1e-3), "unit": "gene-evaluations/s",
                 "full_sweep_seconds_on_this_many_gpus": 44 * N_GENES / (evals / (ms_s * 1e-3)) / world}

    # ---------------- training step (configs[2]): fwd + bwd + AdamW, DP all-reduce ----------
    train = None
    if not args.no_train:
        reg = make_model(ChromoformerRegressor).cuda().train()
        reg.precision = args.train_precision      # the precision the gradient-parity tests cover (tests/test_training_gpu.py)
        tb = synthetic.make_batch(64, ragged=False, seed=100 + rank)
        tdev = {k: ({b: t.to(dev) for b, t in v.items()} if isinstance(v, dict) else v.to(dev)) for k, v in tb.items()}
        target = tdev["labels_reg"].view(-1, 1)
        step = TrainStep(reg, lr=3e-5, regression=True)
        lib.chromo_launch_counter(1)
        step(tdev, target)
        train_launches = int(lib.chromo_launch_counter(1))
        for _ in range(3):                                    # eager steps, then the capture of the chain
            step(tdev, target)
        # the batch lives in the step's own input buffers (where a loader's host->device copies would put it)
        bufs = step.input_buffers(tdev, target)
        tb_, tg_ = bufs if bufs is not None else (tdev, target)
        ms_t = timed(lambda: step(tb_, tg_), 100, 5)
        train = {"metric": "train samples/sec", "value": world * 64 / (ms_t * 1e-3), "unit": "samples/s",
                 "ms_per_step": ms_t, "per_gpu_batch": 64, "model": "Chromoformer-reg", "gpu_launches": train_launches,
                 "dtype": args.train_precision,
                 "collective": "nccl all_reduce of %d fp32 grads" % reg.n_active if world > 1 else "none (1 GPU)",
                 "loss": float(step.loss.item())}

    # ---------------- CPU baseline (rank 0, N = 1 only) -------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref_line = cpu_baseline_subprocess(steps=4, warmup=1, train=not args.no_train)
        cpu = ref_line.get("cpu_baseline") or ref_line
        if train is not None and isinstance(ref_line.get("train"), dict):
            train["cpu_baseline"] = ref_line["train"]
        cpu_getitem = ref_line.get("getitem")
        if cpu_getitem:
            cpu["getitem"] = cpu_getitem

    if rank == 0:
        line = {"metric": "genes/sec inference", "value": genes_per_s, "unit": "genes/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
                "config": workload_config(args), "clocks": clocks, "e2e": e2e,
                "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
                "sustained": sustained, "ragged": ragged,
                "roofline": roofline, "sqa_kernel": sqa_line, "input_path": input_path, "raw_depth_path": raw_path, "ensemble_sweep": sweep, "cpu_baseline": cpu,
                "train": train}
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
