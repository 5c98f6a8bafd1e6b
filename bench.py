"""bench.py — benchmark of the SO-Net forward hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config cfg2]
                    [--dump-outputs DIR]

Default (--config cfg2, BASELINE.json configs[1], the headline): a "step" is one eval-mode
classifier forward (ModelNet40 shape: batch 64 per GPU, N=5000 points, 8x8 SOM, k=3, som_k=9,
fp32) over one batch of synthetic clouds. The other BASELINE.json configs emit the same JSON
shape: cfg1 (classifier B=8 N=1024), cfg3 (ShapeNetPart segmenter forward + per-point logits,
B=32 N=1024), cfg4 (auto-encoder forward + Chamfer, B=32 N=5000). N>1: launched by torchrun, one
rank per GPU, weights replicated, batch sharded (weak scaling), one NCCL all-gather of the step's
result rows per step inside the timed region (issued asynchronously: step i's gather completes
under step i+1's forward; every gather is waited for inside a timed step). Rank 0 prints ONE JSON
line.

  value     clouds/s with inputs resident in HBM (CUDA events per step, L2 flushed between steps,
            max over ranks)
  e2e       the same metric through the public API Model.set_input()/test_model() with pinned
            HOST buffers: every step copies its full inputs host->device and reads its result
            device->host inside the timed region (K steps = K H2D + K D2H). The loop is a serving
            loop pipelined by call order only: set_input (async, double-buffered, copy stream) +
            test_model + async D2H of step i+1 are issued before the host waits for step i
  roofline  dominant kernel (by measured device time) vs MEASURED_PEAKS.json, measured live with
            CUDA events around every C-ABI call of instrumented steps; `kernels` lists all of
            them; `roofline.secondary`: the standalone HBM-bound ops (index_max, query_topk)
  cpu_baseline   the reference's own PyTorch-CPU path — its unmodified Model class from the
            bytecode build product oracle/_ref/pyref, pool in its own compiled plugin ("kind":
            "reference"; the oracle port only if that cannot be imported) — timed on this box's
            host cores on a bounded sample (8 clouds of this run's inputs). Its outputs are also
            the parity check of the timed GPU steps ("parity")
  --impl reference   only that CPU arm, same JSON shape with "impl": "reference"
  --dump-outputs DIR   after the timed steps, rank 0 writes what the last timed step handed its
            caller (the task's Model outputs, step_outputs()) as DIR/<name>.npy, float32. Inputs
            and weights are seeded, so two builds run with the same arguments can be compared
            array by array.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "so-net_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

UNIT = "clouds/s"
M_NODES, SOM_K, K_NN = 64, 9, 3
CONFIGS = {
    "cfg2": dict(task="classifier", B=64, N=5000,
                 metric="point-clouds/sec forward (ModelNet40 5000pt, 8x8 SOM)",
                 workload="ModelNet40 classifier forward, batch=64/GPU, N=5000 pts, 8x8 SOM, k=3, "
                          "som_k=9, fp32, eval (BASELINE.json configs[1])"),
    "cfg1": dict(task="classifier", B=8, N=1024,
                 metric="point-clouds/sec forward (ModelNet40 1024pt, 8x8 SOM)",
                 workload="ModelNet40 classifier forward, batch=8/GPU, N=1024 pts, 8x8 SOM, k=3, "
                          "som_k=9, fp32, eval (BASELINE.json configs[0])"),
    "cfg3": dict(task="segmenter", B=32, N=1024,
                 metric="point-clouds/sec forward + per-point logits (ShapeNetPart 1024pt, 8x8 SOM)",
                 workload="ShapeNetPart segmenter forward + per-point logits [B,50,N], batch=32/GPU, "
                          "N=1024 pts, 8x8 SOM, k=3, som_k=9, fp32, eval (BASELINE.json configs[2])"),
    "cfg4": dict(task="autoencoder", B=32, N=5000,
                 metric="point-clouds/sec forward + Chamfer (auto-encoder 5000pt, 8x8 SOM)",
                 workload="Auto-encoder forward (encoder + FC/up-conv decoder, 1280 predicted points) + "
                          "Chamfer(256 vs 5000) + Chamfer(1280 vs 5000), batch=32/GPU, N=5000 pts, 8x8 "
                          "SOM, fp32, eval (BASELINE.json configs[3])"),
}
METRIC = CONFIGS["cfg2"]["metric"]
WORKLOAD = CONFIGS["cfg2"]["workload"]
# dram__bytes_read.sum + dram__bytes_write.sum per launch at the cfg2 workload, from the committed
# `ncu --set full` captures (profiles/); None until a capture exists.
NCU_TRAFFIC = {"index_max_f32": 1.4871e9,
               # profiles/r01h_pointresnet_tc_pool_compact.ncu-rep: 33.89 MB read + 2.8 KB written
               "pointresnet_tc_pool_forward": 33.895e6,
               # profiles/r02d_query_topk.ncu-rep: 3.92 MB read + 198.3 MB written (245.8 MB
               # algorithmic: part of the mask was still in L2 when the capture ended)
               "query_topk": 202.26e6}
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            d["_source"] = "measured"
            return d
        except Exception:
            pass
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


# ---- clocks sampling (B200_PROFILING.md recipe) -----------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "samples": len(sm),
                "reasons": sorted(reasons)}


# ---- task adapters: one table for the GPU arm (sonet_b200) and the CPU arm (the reference) ---------
def head_name(task):
    return {"classifier": "classifier", "segmenter": "segmenter", "autoencoder": "decoder"}[task]


def make_states(task, B, N):
    """Seeded weights (CPU tensors, reference state_dict keys): encoder seed 1, head seed 2."""
    from sonet_b200 import networks, synth
    opt = synth.make_opt(task, batch_size=B, input_pc_num=N)
    head = {"classifier": networks.Classifier, "segmenter": networks.Segmenter,
            "autoencoder": networks.Decoder}[task](opt)
    return (synth.synth_state_dict(networks.Encoder(opt), seed=1),
            synth.synth_state_dict(head, seed=2))


def input_list(task, inp, B, N):
    """set_input arguments of the task's Model (models/{classifier,segmenter,autoencoder}.py)."""
    if task == "segmenter":
        seg = inp.get("seg")
        if seg is None:
            seg = inp["seg"] = (torch.arange(B * N, dtype=torch.int64).view(B, N) * 7) % 50
        return [inp["pc"], inp["sn"], inp["label"], seg, inp["node"], inp["node_knn_I"]]
    return [inp["pc"], inp["sn"], inp["label"], inp["node"], inp["node_knn_I"]]


def result_rows(task, model):
    """The per-cloud result of a step: what is all-gathered, read back and parity-checked."""
    if task == "classifier":
        return model.score                                   # [B, classes]
    if task == "segmenter":
        return model.score_segmenter                         # [B, 50, N]
    return torch.stack((model.chamfer_criteria.forward_loss_array,
                        model.chamfer_criteria.backward_loss_array), dim=1)   # [B, 2]


DUMP_BUDGET = 64 << 20       # bytes that --dump-outputs writes, all arrays together


def step_outputs(task, model):
    """What a caller reads from the Model after test_model() (models/<task>.py), as float32
    host copies."""
    names = {"classifier": ("score", "feature", "loss"),
             "segmenter": ("score_segmenter", "feature", "loss"),
             "autoencoder": ("predicted_pc", "feature", "loss_chamfer", "loss_chamfer_conv4",
                             "loss")}[task]
    out = {n: getattr(model, n) for n in names if torch.is_tensor(getattr(model, n, None))}
    if task == "autoencoder":
        out["chamfer_loss_arrays"] = result_rows(task, model)
    return {n: t.detach().float().cpu() for n, t in out.items()}


def dump_outputs(path, arrays):
    """Write each array as <path>/<name>.npy. An array larger than its share of DUMP_BUDGET is
    written as a sample of its flattened elements at positions drawn from a fixed seed, so that
    two runs sample the same positions."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    share = DUMP_BUDGET // (4 * len(arrays))                  # float32 elements per array
    for name, t in arrays.items():
        if t.numel() > share:
            g = torch.Generator().manual_seed(0)
            t = t.reshape(-1)[torch.randperm(t.numel(), generator=g)[:share].sort().values]
        np.save(os.path.join(path, name + ".npy"), t.numpy())


# ---- CPU arm: the reference's own PyTorch-CPU path ---------------------------------------------------
def _cpu_step_fn(cfg, sample_B, inp, st_e, st_h):
    """Returns (step() -> result rows [sample_B, ...], set_threads(n), kind, description).

    kind "reference": the UNMODIFIED reference — its own models/<task>.py Model (set_input +
    test_model, exactly the calls of modelnet/train.py:72-76) on its own networks/layers/som/losses
    modules, imported from the bytecode build product oracle/_ref/pyref (or /root/reference where
    that exists) with the shims of oracle/ref_shims.py; the pool runs in the reference's own
    compiled plugin (forward_multi_thread_cpu, its faster CPU variant); Chamfer's Faiss search is
    the exact brute-force stub (Faiss is not vendored).
    kind "port": the oracle restatement (oracle/oracle.py), only when the reference cannot be
    imported on this machine."""
    from sonet_b200 import synth
    task, N = cfg["task"], cfg["N"]
    opt = synth.make_opt(task, batch_size=sample_B, input_pc_num=N)
    args = input_list(task, inp, sample_B, N)
    try:
        from oracle import ref_shims
        ref = ref_shims.install(prefer_pyref=True, pool_threads=os.cpu_count() or 1)
        with ref_shims.cpu_only():       # the SOM node buffer follows cuda availability, not opt.device
            model = getattr(ref, task).Model(opt)
        model.encoder.load_state_dict(st_e)
        getattr(model, head_name(task)).load_state_dict(st_h)
        binary = bool(getattr(ref.index_max, "is_reference_binary", False))

        def step():
            model.set_input(*args)
            model.test_model()
            return result_rows(task, model).detach()

        def set_threads(n):
            torch.set_num_threads(n)
            ref.index_max.pool_threads = n
        where = "oracle/_ref/pyref bytecode" if ref.root != ref_shims.REF else "/root/reference"
        return step, set_threads, "reference", (
            "reference %s.Model.set_input/test_model from %s; index_max via %s"
            % (task, where, "the reference's compiled forward_multi_thread_cpu" if binary
               else "the C restatement (reference plugin not built)"))
    except Exception as e:                                   # noqa: BLE001
        why = "%s: %s" % (type(e).__name__, e)
    from oracle import oracle
    threads = {"n": os.cpu_count() or 1}

    def step():
        with torch.no_grad():
            o = oracle.encoder_forward(st_e, opt, inp["pc"], inp["sn"], inp["node"],
                                       inp["node_knn_I"], fast_pool=threads["n"])
            if task == "classifier":
                return oracle.classifier_forward(st_h, o["feature"])
            if task == "segmenter":
                return oracle.segmenter_forward(st_h, opt, o, inp["pc"], inp["sn"], inp["label"])
            raise RuntimeError("no oracle port of the auto-encoder decoder (%s)" % why)

    def set_threads(n):
        torch.set_num_threads(n)
        threads["n"] = n
    return step, set_threads, "port", "oracle port (reference not importable here: %s)" % why


def cpu_arm(cfg, steps, warmup, sample_B=8, inp=None):
    """Time the reference's CPU path on the host cores, on a bounded sample (sample_B clouds of
    the config's shape). Returns the cpu_baseline dict and the result rows of the sample."""
    from oracle import build as obuild
    obuild.build_c()
    from sonet_b200 import synth
    cores = os.cpu_count() or 1
    sample_B = min(sample_B, cfg["B"])
    st_e, st_h = make_states(cfg["task"], sample_B, cfg["N"])
    if inp is None:
        inp = synth.synth_inputs(sample_B, cfg["N"], seed=0)
    step, set_threads, kind, desc = _cpu_step_fn(cfg, sample_B, inp, st_e, st_h)

    # the reference path does not scale to every core count: probe a few thread counts and time
    # the best one (the faster reference number is the one compared against, SURVEY.md §8d)
    probe = {}
    for n in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)},
                    reverse=True):
        set_threads(n)
        step()
        t0 = time.perf_counter()
        step()
        probe[n] = time.perf_counter() - t0
    best = min(probe, key=probe.get)
    set_threads(best)
    for _ in range(max(warmup - 1, 0)):
        step()
    times = []
    rows = None
    for _ in range(steps):
        t0 = time.perf_counter()
        rows = step()
        times.append(time.perf_counter() - t0)
    per = sum(times) / len(times)
    return dict(value=sample_B / per, unit=UNIT, cores=best, host_cores=cores,
                kind=kind, ms_per_step=per * 1e3,
                thread_probe_s={str(k): round(v, 3) for k, v in probe.items()},
                sample="%d steps of a B=%d x N=%d %s forward (%s), best of the probed "
                       "thread counts, after warm-up" % (steps, sample_B, cfg["N"], cfg["task"],
                                                         desc)), rows


def run_reference_arm(args, rank, cfg):
    if rank != 0:
        return
    steps = args.steps
    warm = max(1, min(args.warmup, 2))
    cb, _ = cpu_arm(cfg, steps, warm)
    line = {"impl": "reference", "metric": cfg["metric"], "value": cb["value"], "unit": UNIT,
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": cb["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": cfg["workload"],
                                            "sample_batch": min(8, cfg["B"])},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---- per-kernel roofline from instrumented steps -----------------------------------------------------
def kernel_report(profile_steps, peaks):
    """profile_steps: list of lists of (name, e0, e1, args). Returns per-call-site rows."""
    rows = {}
    order = []
    for prof in profile_steps:
        seen = {}
        for name, e0, e1, a in prof:
            ms = e0.elapsed_time(e1)
            i = seen.get(name, 0)
            seen[name] = i + 1
            key = "%s#%d" % (name.replace("sonet_", ""), i)
            if key not in rows:
                rows[key] = dict(name=key, ms=[], args=a)
                order.append(key)
            rows[key]["ms"].append(ms)
    out = []
    # per-kernel rows: each kernel is timed alone between CUDA events in a short eager pass at full
    # boost clocks -> the BURST bf16 peak is the denominator (MEASURED_PEAKS.json "bf16_tflops")
    hbm, tf = peaks["hbm_gbs"], peaks["bf16_tflops"]
    for key in order:
        r = rows[key]
        ms = sum(r["ms"]) / len(r["ms"])
        a = r["args"]
        row = {"kernel": key, "ms": round(ms, 4)}
        if key.startswith("pointwise_layer"):
            C0, C1, B, P, Cout = a[1], a[3], a[4], a[5], a[9]
            flops = 2.0 * B * P * (C0 + C1) * Cout
            ach = flops / (ms * 1e-3) / 1e12
            row.update(bound="tensor", achieved=round(ach, 3), peak=tf, unit="TFLOP/s",
                       frac=round(ach / tf, 5), shape="[%d,%d+%d,%d]->%d" % (B, C0, C1, P, Cout),
                       note="fp32 CUDA-core path vs the bf16 tensor peak")
        elif key.startswith("pointwise_tc_forward"):
            # args of sonet_pointwise_tc_forward: x0, C0, x1, C1, B, P, blob, inv, shift, Cout, ...
            C0, C1, B, P, Cout = a[1], a[3], a[4], a[5], a[9]
            flops = 2.0 * B * P * (C0 + C1) * Cout
            ach = flops / (ms * 1e-3) / 1e12
            row.update(bound="tensor", achieved=round(ach, 2), peak=tf, unit="TFLOP/s",
                       frac=round(ach / tf, 4), executed_tflops=round(3 * ach, 1),
                       shape="[%d,%d+%d,%d]->%d" % (B, C0, C1, P, Cout),
                       note="algorithmic flops (x3 executed: fp16 hi/lo split); the CUDA-event time of "
                            "a 30-70 us launch includes host launch latency in this eager pass")
        elif key.startswith("pointresnet_tc_forward") or key.startswith("pointresnet_tc_pool_forward"):
            Bc, P = a[2], a[3]
            flops = 328448.0 * Bc * P          # SURVEY §8d: 2 * (6*64 + 64*128 + 128*256 + 320*384)
            ach = flops / (ms * 1e-3) / 1e12
            row.update(bound="tensor", achieved=round(ach, 2), peak=tf, unit="TFLOP/s",
                       frac=round(ach / tf, 4), executed_tflops=round(3 * ach, 1),
                       shape="[%d,%d,%d] 6->64->128->256->[320]->384" % (Bc, a[1], P),
                       note="algorithmic flops; the fp16 hi/lo split executes 3x as many on "
                            "the tensor pipe, so frac <= 0.33 by construction"
                            + ("; per-node max fused into the epilogue (first_pn_out never "
                               "written)" if "pool" in key else ""))
        elif key.startswith("index_max"):
            B, C, N, K = a[2], a[3], a[4], a[5]
            byts = 4.0 * B * C * N + 4.0 * B * N + 4.0 * B * C * K * (2 if a[7] else 1)
            ach = byts / (ms * 1e-3) / 1e9
            row.update(bound="hbm", achieved=round(ach, 1), peak=hbm, unit="GB/s",
                       frac=round(ach / hbm, 4), shape="[%d,%d,%d] K=%d" % (B, C, N, K))
        elif key.startswith("som_mask"):
            B, kN, M = a[1], a[2], a[3]
            byts = 4.0 * B * kN * M + 4.0 * B * kN
            ach = byts / (ms * 1e-3) / 1e9
            row.update(bound="hbm", achieved=round(ach, 1), peak=hbm, unit="GB/s",
                       frac=round(ach / hbm, 4))
        out.append(row)
    return out


def fused_kernel_clock(model, dev):
    """SM clock the fused tcgen05 kernel actually runs at: SM cycles counted by CTA 0 (clock64, the
    kernel's debug timeline entry point) against the CUDA-event duration of the same launch.
    nvidia-smi's samples (>= 20 ms apart) cannot see inside a 0.7 ms kernel; under tensor load the
    chip is power-managed below clocks.max.sm within the kernel."""
    from sonet_b200 import _C, ops, synth
    B, N, M = 64, 5000, M_NODES
    try:
        inp = synth.synth_inputs(B, N, seed=0)
        pc, sn, node = inp["pc"].to(dev), inp["sn"].to(dev), inp["node"].to(dev)
        a = ops.som_assign(pc, node, K_NN)
        xs, ns, p0i = ops.som_sort_decenter(pc, sn, a["cluster_mean"], a["min_idx_i32"], a["count"], K_NN)
        blob, fpar = model.encoder.first_pointnet._tc_params()
        keys = torch.empty(B, 384, M, dtype=torch.int32, device=dev)
        _C.check(_C.lib().sonet_pool_keys_init(keys.data_ptr(), keys.numel(), None), "init")
        p0 = torch.empty(B, 384, device=dev)
        tl = torch.zeros(128, dtype=torch.int64, device=dev)
        tl[125] = 3
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        torch.cuda.synchronize()
        for i in range(4):
            if i == 3:
                ev[0].record()
            _C.check(_C.lib().sonet_debug_pointresnet_tc_pool_timeline(
                xs.data_ptr(), 6, B, K_NN * N, blob.data_ptr(), fpar.data_ptr(), ns.data_ptr(),
                p0i.data_ptr(), M, keys.data_ptr(), p0.data_ptr(), tl.data_ptr(), None), "timeline")
        ev[1].record()
        torch.cuda.synchronize()
        t = tl.cpu().tolist()
        cycles = t[64 + 63] - t[64 + 62]
        ms = ev[0].elapsed_time(ev[1])
        return {"sm_cycles_cta0": cycles, "ms": round(ms, 4), "sm_mhz_in_kernel": round(cycles / ms / 1e3, 1)}
    except Exception as e:                                  # noqa: BLE001  (diagnostic only)
        return {"error": "%s: %s" % (type(e).__name__, e)}


def standalone_rows(model, cfg, peaks, dev, flush):
    """HBM-bound API ops that no longer run inside the classifier step (the max is fused into the
    MLP epilogue, the dense mask is never built): timed standalone on the cfg2 tensors."""
    from sonet_b200 import ops
    from sonet_b200 import som as som_mod
    B, NPTS = 64, 5000
    g = torch.Generator(device=dev).manual_seed(0)
    data = torch.randn(B, 384, K_NN * NPTS, device=dev, generator=g)
    index = torch.randint(0, M_NODES, (B, K_NN * NPTS), device=dev, generator=g, dtype=torch.int32)

    def time_op(fn, reps=5, rounds=4):
        """CUDA-event time of `reps` back-to-back launches (host launch latency hidden behind
        the L2 flush write), averaged; working sets exceed L2 so every launch streams HBM."""
        for _ in range(3):
            fn()
        ts = []
        for _ in range(rounds):
            flush.zero_()
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / reps)
        return sum(ts) / len(ts)

    out = []
    ms_im = time_op(lambda: ops.index_max(data, index, M_NODES, with_values=True))
    byts = 4.0 * B * 384 * K_NN * NPTS + 4.0 * B * K_NN * NPTS + 8.0 * B * 384 * M_NODES
    out.append({"kernel": "index_max_f32 (standalone, [64,384,15000] K=64)",
                "ms": round(ms_im, 4), "bound": "hbm",
                "achieved": round(byts / (ms_im * 1e-3) / 1e9, 1),
                "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(byts / (ms_im * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                "traffic": NCU_TRAFFIC.get("index_max_f32")})
    del data, index
    # SOM kNN with the API-complete outputs of BatchSOM.query_topk (util/som.py:237-269): top-k
    # assignment + int64 indices + the dense one-hot mask [B,kN,M] int32 (245 MB): HBM-bound
    from sonet_b200 import synth
    inp = synth.synth_inputs(B, NPTS, seed=0)
    pc = inp["pc"].to(dev)
    bs = som_mod.BatchSOM(8, 8, 3, dev.index or 0, B)
    bs.node = inp["node"].to(dev)
    ms_q = time_op(lambda: bs.query_topk(pc, K_NN))
    kN = K_NN * NPTS
    byts = B * (12.0 * NPTS + 12.0 * M_NODES + 8.0 * kN + 4.0 * M_NODES + 4.0 * kN * M_NODES)
    out.append({"kernel": "BatchSOM.query_topk (top-k assignment + dense mask + row_max, one launch), "
                          "B=64 N=5000",
                "ms": round(ms_q, 4), "bound": "hbm",
                "achieved": round(byts / (ms_q * 1e-3) / 1e9, 1),
                "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(byts / (ms_q * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                "traffic": NCU_TRAFFIC.get("query_topk")})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="sonet_b200", choices=["sonet_b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS),
                    help="BASELINE.json config (cfg2 = configs[1], the headline)")
    ap.add_argument("--collective", default="torch", choices=["torch", "sonet"],
                    help="N>1: all-gather through torch.distributed (NCCL) or through the C-ABI "
                         "sonet_allgather (the same NCCL, resolved by libsonet_b200)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager op calls instead of CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    cfg = CONFIGS[args.config]
    task, B, NPTS = cfg["task"], cfg["B"], cfg["N"]

    from sonet_b200 import dist as sdist
    rank, local_rank, world = sdist.env_world()
    if args.impl == "reference":
        run_reference_arm(args, rank, cfg)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference "
                         "for the CPU arm")
    rank, local_rank, world = sdist.init_from_env()
    dev = torch.device("cuda", torch.cuda.current_device())
    import importlib

    import torch.distributed as dist
    from sonet_b200 import _C, ops, synth
    _C.lib()
    peaks = load_peaks()

    opt = synth.make_opt(task, batch_size=B, input_pc_num=NPTS, device=str(dev), gpu_id=dev.index)
    model = importlib.import_module("sonet_b200." + task).Model(opt)
    st_e, st_h = make_states(task, B, NPTS)
    model.encoder.load_state_dict(st_e)
    getattr(model, head_name(task)).load_state_dict(st_h)
    if not args.no_graph:
        model.enable_cuda_graph(True)                      # one graph launch per step
    inp = synth.synth_inputs(B, NPTS, seed=rank)            # each rank: its own shard
    host = [t.pin_memory() for t in input_list(task, inp, B, NPTS)]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host)
    total_rows = B * world

    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- the step: forward (+ asynchronous all-gather of its result rows) ----------------------------
    model.set_input(*host)
    model.test_model()
    row_shape = tuple(result_rows(task, model).shape[1:])
    d2h_bytes = B * int(torch.tensor(row_shape).prod()) * 4
    ag = sdist.AsyncGather(world, (B,) + row_shape, dev, impl=args.collective) if world > 1 else None
    gathered = ag.out if ag else None

    def gpu_step(i):
        """Forward i; its result rows are staged (the graph's static buffer is overwritten by the
        next replay) and all-gathered ASYNCHRONOUSLY; the gather of step i-1, which ran under this
        forward, is waited for before the step ends — every gather completes inside a timed step."""
        model.test_model()
        rows = result_rows(task, model)
        if world == 1:
            return rows
        o = ag.launch(i, rows)
        ag.wait_prev(i)
        return o

    def drain():
        if ag:
            ag.drain()

    # ---- (1) device-resident arm -------------------------------------------------------------------
    torch.cuda.synchronize()
    # rank 0 only: eight nvidia-smi pollers hitting the driver while every timed step contains a
    # cross-rank all-gather turn one rank's stall into everybody's
    sampler = ClockSampler(dev.index)
    if rank == 0:
        sampler.start()                                    # runs through both timed regions
    for i in range(args.warmup):
        gpu_step(i)
    drain()
    time.sleep(0.3)                                        # let nvidia-smi deliver its first sample
    for i in range(args.warmup):
        gpu_step(i)
    drain()
    barrier()
    l0 = ops.KERNEL_LAUNCHES
    evs = []
    wall0 = time.perf_counter()
    out = None
    for i in range(args.steps):
        flush.zero_()                                      # L2 flush, outside the event pair
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = gpu_step(i)
        if i == args.steps - 1:
            drain()                                        # the last gather also ends inside a timed step
        e1.record()
        evs.append((e0, e1))
    barrier()
    wall = time.perf_counter() - wall0
    timed_rows = result_rows(task, model).detach().clone()  # result of the last timed step
    timed_gather = out.detach().clone()
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = step_outputs(task, model)
        if world > 1:
            dumped["gathered_rows"] = timed_gather.float().cpu()
    launches = ops.KERNEL_LAUNCHES - l0
    step_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    ms_per_step = total_ms / args.steps
    value = total_rows * args.steps / (total_ms * 1e-3)

    # multi-GPU parity (outside every timed region): the gathered rows of this rank's shard are
    # bit-identical to what it computed, and rank 0 recomputes rank 1's shard locally (same
    # seeded inputs and weights): gathered rows == a single-GPU run, bit for bit (SURVEY §8e)
    gather_check = None
    if world > 1:
        own_ok = bool(torch.equal(timed_gather[rank * B:(rank + 1) * B], timed_rows))
        flag = torch.tensor([1 if own_ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        other_ok = None
        if rank == 0:
            inp1 = synth.synth_inputs(B, NPTS, seed=1)
            model.set_input(*input_list(task, inp1, B, NPTS))
            model.test_model()
            other_ok = bool(torch.equal(result_rows(task, model), timed_gather[B:2 * B]))
            model.set_input(*host)
            model.test_model()
        gather_check = {"own_shard_bit_identical_all_ranks": bool(flag.item() == 1),
                        "rank1_shard_recomputed_on_rank0_bit_identical": other_ok}
        if not gather_check["own_shard_bit_identical_all_ranks"] or other_ok is False:
            raise SystemExit("bench.py: gathered rows differ from the per-rank results: %s" % gather_check)

    # ---- (2) end-to-end arm: host buffers through the public Model API ------------------------------
    # A serving loop over the public API, software-pipelined by call order only: the (async,
    # double-buffered, copy-stream) set_input of batch i+1 is issued before the result of batch i
    # is read back. Every step still copies its full inputs host->device (from pinned memory) and
    # reads its result rows device->host inside the timed region; K steps = K H2D + K D2H.
    pinned_out = [torch.empty((total_rows,) + row_shape, dtype=torch.float32).pin_memory()
                  for _ in range(2)]
    out_ready = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_run(k_steps):
        def launch(i):                    # H2D + forward (+ all-gather) + async D2H of step i
            model.set_input(*host)
            model.test_model()
            o = result_rows(task, model)
            if world > 1:
                dist.all_gather_into_tensor(gathered[i & 1], o.contiguous())
                o = gathered[i & 1]
            pinned_out[i & 1].copy_(o, non_blocking=True)
            out_ready[i & 1].record()
        launch(0)
        last = None
        for i in range(k_steps):
            if i + 1 < k_steps:
                launch(i + 1)                              # keep the GPU fed
            out_ready[i & 1].synchronize()                 # result of step i is on the host
            last = pinned_out[i & 1]
        return last
    e2e_run(args.warmup)
    barrier()
    flush.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    t_e2e = [time.perf_counter() - t0]
    barrier()
    e2e_total = torch.tensor([sum(t_e2e)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_total, op=dist.ReduceOp.MAX)
    e2e_value = total_rows * args.steps / float(e2e_total.item())
    clocks = sampler.stop()

    # ---- (3) instrumented steps: per-kernel device time with CUDA events ---------------------------
    prof_steps = []
    model.enable_cuda_graph(False)                         # per-kernel events need eager calls
    for _ in range(3):
        flush.zero_()
        ops.PROFILE = []
        model.test_model()
        torch.cuda.synchronize()
        prof_steps.append(ops.PROFILE)
        ops.PROFILE = None
    kernels = kernel_report(prof_steps, peaks)
    kernel_ms = sum(r["ms"] for r in kernels)
    # the dominant kernel = the launch with the largest measured device time among those with a
    # roofline model (the fused tcgen05 PointResNet on the default path)
    modelled = [r for r in kernels if "bound" in r]
    dom = max(modelled, key=lambda r: r["ms"])
    roofline = {"kernel": dom["kernel"], "bound": dom["bound"], "achieved": dom["achieved"],
                "peak": dom["peak"], "unit": dom["unit"], "frac": dom["frac"],
                "traffic": NCU_TRAFFIC.get(dom["kernel"].split("#")[0]) if args.config == "cfg2" else None,
                "peak_source": peaks["_source"] + (" bf16 burst (kernel timed alone)"
                                                   if dom["bound"] == "tensor"
                                                   else " copy bandwidth"),
                "ms": dom["ms"], "share_of_step": round(dom["ms"] / kernel_ms, 4),
                "note": dom.get("note")}

    standalone = standalone_rows(model, cfg, peaks, dev, flush) if rank == 0 else []
    if rank == 0 and args.config == "cfg2" and dom["kernel"].startswith("pointresnet_tc_pool"):
        # the dominant kernel is power-managed below the nominal clock: report the clock it ran
        # at and its EXECUTED tensor rate against the sustained (seconds-long, power-capped) peak
        ck = fused_kernel_clock(model, dev)
        roofline["clock_in_kernel"] = ck
        sustained = peaks.get("bf16_tflops_sustained")
        if sustained and "executed_tflops" in dom:
            roofline["executed_tflops"] = dom["executed_tflops"]
            roofline["executed_frac_of_sustained_peak"] = round(dom["executed_tflops"] / sustained, 4)

    # CPU leg (rank 0, N=1): the reference's own CPU path on the first 8 clouds of THIS run's
    # inputs with THIS run's weights — timed as the cpu_baseline, and its result rows double as the
    # parity check of the rows the timed GPU steps produced (outside every timed region)
    cpu_baseline, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sb = min(8, B)
        sample = {k: v[:sb].contiguous() for k, v in inp.items()}
        cpu_baseline, ref_rows = cpu_arm(cfg, steps=3, warmup=1, sample_B=sb, inp=sample)
        got = timed_rows[:sb].cpu()
        err = float(((got - ref_rows).abs() / ref_rows.abs().clamp(min=1.0)).max())
        tol = 1e-4
        parity = {"parity_checked": True, "against": cpu_baseline["kind"],
                  "what": "result rows of the timed steps (graph replay) for clouds 0-%d vs the CPU "
                          "arm's on the same inputs/weights" % (sb - 1),
                  "max_rel_err": err, "tol": tol, "ok": err <= tol}
        if not parity["ok"]:
            raise SystemExit("bench.py: GPU results differ from the CPU reference: %.3e" % err)

    if rank == 0:
        line = {"metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": cfg["workload"], "name": args.config,
                           "global_batch": total_rows,
                           "parallelism": "dp%d batch-sharded, 1 async all-gather of the result rows/step "
                                          "(%s)" % (world, args.collective),
                           "l2": "256 MB flush write between timed steps (outside event pairs)",
                           "weights": "random (seeded), BN stats randomised",
                           "launch": "eager" if args.no_graph else
                                     "CUDA-graph replay of the step (Model.enable_cuda_graph)"},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                        "d2h_bytes_per_step": d2h_bytes * world},
                "gpu_launches": launches, "wall_s_timed_region": round(wall, 4),
                "step_ms": {"min": round(min(step_ms), 4), "median": round(statistics.median(step_ms), 4),
                            "max": round(max(step_ms), 4)},
                "clocks": clocks,
                "roofline": dict(roofline, secondary=standalone), "kernels": kernels,
                "cpu_baseline": cpu_baseline,
                "parity": parity,
                "parity_checked": bool(parity and parity["ok"]),
                "gather_check": gather_check,
                "checksum": float(timed_gather.double().sum().item())}
        if dumped:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
