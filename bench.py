#!/usr/bin/env python
"""bench.py -- fake-quant hot-path throughput (BASELINE.json metric) on B200.

A "step" is one pass of the hot path over one batch of synthetic input: every activation
fake-quant call of ONE VAR generation pass (10 stages x depth blocks x 4 quantized linears,
fpqvar_b200/var_workload.py).  Default workload = BASELINE.json configs[2], the configuration
the metric is quoted on (VAR-d30 256x256 W4A4 fp_e2 + fc2 fp_e1m2_neg_e2m1_pos, block rotate +
GALT transform, B=50 per GPU).  Multi-GPU: image batches are independent, so every rank runs its
own batch (weak scaling, no data-path collective; one final gather of the timings).

  value     algorithmic GB/s (input bytes read once + output bytes written once), inputs resident
            in HBM, one CUDA-graph replay per step, CUDA events, max over ranks
  e2e       same metric through the HOST-buffer entry (fpqvar_b200.hotpath.HostPipeline): pinned
            H2D copy of every input and D2H copy of every output inside the timed region; every rank
            binds to its GPU's NUMA node before it allocates its pinned buffers
  roofline  the dominant kernel's launches of the step, timed alone with CUDA events; `traffic` from
            the committed ncu capture (profiles/r2_traffic.json)
  cpu_baseline   the reference's OWN torch CPU functions (baseline/_ref, installed by
            baseline/install_ref.sh; kind "reference") on a bounded sample of the same workload, rank 0 /
            N=1 only; `cpu_port` = the multi-threaded C port of the oracle beside it.  Without an install:
            the port (kind "port")
  reference_gpu_path / generation_reference_model   the reference's own GPU path (its fp_quant_*_cuda functions
            around its extension compiled for sm_100a) over the same step, and images/sec of the reference's
            own VAR model with its quantizers / this library as a drop-in / the fused call sites -- child
            processes, outside every timed region
  search    BASELINE configs[4] on a bounded unit list, (layer, weight-format) units sharded over the ranks,
            one all-reduce (strong scaling)
  other_configs   the device-resident step of BASELINE configs[1] and [3] (child runs)

`--impl reference` times the reference's CPU implementation alone, on this arm's config / metric / unit, with
the steps and warm-up it is given (rank 0 only under torchrun).
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fake-quant GB/s over the hot path of one VAR generation pass (config.workload; % of HBM peak = roofline.frac)"
UNIT = "GB/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="var_d30_w4a4_rot")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-generation", action="store_true",
                    help="skip the images/sec leg (tools/var_generate.py: a full VAR generation pass around the hot path)")
    ap.add_argument("--gen-iters", type=int, default=3)
    ap.add_argument("--no-search", action="store_true", help="skip the format-search leg (BASELINE configs[4] on a bounded unit list)")
    ap.add_argument("--search-blocks", type=int, default=2, help="transformer blocks whose four layers the search leg scores (the full sweep has 30)")
    ap.add_argument("--no-lowbit", action="store_true", help="skip the low-bit GEMM leg (SURVEY section 8 f4)")
    ap.add_argument("--no-reference-legs", action="store_true",
                    help="skip reference_gpu_path / generation_reference_model (the unmodified reference from baseline/_ref on this GPU)")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="skip the short device-resident runs of the other BASELINE configs (other_configs)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--sample-stages", type=int, default=0,
                    help="CPU legs only: restrict the bounded sample to the first N stages (0 = all; used by the CPU unit test)")
    ap.add_argument("--profile", action="store_true",
                    help="for ncu: one warm-up replay + the timed steps only (no roofline graphs, no e2e, no CPU baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed seeded sample of every call's output of the last step (rank 0) "
                         "as DIR/s<stage>_<site>.npy, float32 [depth, samples], to compare two builds output for output.  The output arena "
                         "holds only the last 2 GiB of a step's output: every earlier call is launched once more, eagerly, on its "
                         "input, so a defect that shows only under graph capture can be missing from those")
    return ap.parse_args()


def bench_config(hot, world):
    """The `config` object of the JSON line; identical in both arms (--impl b200 / --impl reference)."""
    calls = hot.calls()
    step_bytes = sum(c.bytes for c in calls)
    bits = 6 if hot.act_fmt in ("e2m3", "e3m2") else 4
    return {
        "workload": hot.name,
        "desc": f"VAR-d{hot.depth} W{bits}A{bits} hot path: {len(calls)} activation fake-quant calls of one generation pass, B={hot.batch}/GPU "
                f"({hot.elems_per_pass() / 1e9:.2f} G elements, {step_bytes / 1e9:.1f} GB algorithmic per GPU per step)",
        "l2": "inputs/outputs rotate through 2 GiB/1 GiB/2 GiB/2 GiB arenas (>> 126 MB L2); no address is re-read within 1 GiB of traffic",
        "launch": "one CUDA-graph replay per step", "parallelism": f"dp{world} (independent image batches, no data-path collective)",
    }


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.proc = None
        self.path = f"/tmp/fpq_clocks_{os.getpid()}.csv"
        exe = shutil.which("nvidia-smi")
        if exe:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen([exe, "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as f:
            for line in f:
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 7:
                    continue
                try:
                    sm.append(float(parts[0])); mx.append(float(parts[1]))
                except ValueError:
                    continue
                for n, v in zip(names, parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU baseline / reference arm (oracle port; the ONLY place bench.py touches oracle/)
# ----------------------------------------------------------------------------------------------
def cpu_sample_inputs(hot, np, seed=0, stages=0):
    """Bounded sample: the four quantizer calls of ONE block (of `depth`) at every one of the 10
    stages, i.e. 1/depth of a step."""
    rng = np.random.default_rng(seed)
    calls = [c for c in hot.calls(blocks=[0]) if not stages or c.stage < stages]
    data = []
    for c in calls:
        x = rng.standard_normal((c.rows, c.cols), dtype=np.float32)
        if c.site == "fc2":
            x = 0.5 * x * (1.0 + np.tanh(0.7978845608 * (x + 0.044715 * x ** 3)))     # GELU(tanh) skew, as the fc2 input has
        if c.in_dtype == "f16":
            x = x.astype(np.float16)
        data.append(x)
    return calls, data


def cpu_run_sample(calls, data, smooth, P):
    for c, x in zip(calls, data):
        if c.op == "group":
            P.fake_quant(x, c.fmt, 128, "kernel", out_dtype={"f32": "float32", "f16": "float16"}[c.out_dtype])
        elif c.op == "signsplit":
            P.fake_quant_signsplit(x, c.fmt, 128, "kernel")
        elif c.op == "mod_rotate_quant":
            # the adaLN modulate in front of it (basic_var.py:263): numpy on the [B, rows_per_batch, C] view
            b = c.rows // c.rows_per_batch
            xm = x.reshape(b, c.rows_per_batch, c.cols) * MOD_GAIN[:b, None, :c.cols] + MOD_SHIFT[:b, None, :c.cols]
            P.transform_rotate_quant(xm.reshape(c.rows, c.cols), smooth, c.fmt)
        else:
            P.transform_rotate_quant(x, smooth, c.fmt)


MOD_GAIN = MOD_SHIFT = None


def cpu_baseline(hot, seconds, steps=None, warmup=1, stages=0):
    import numpy as np
    from oracle import port as P       # test infrastructure, used here as the timed CPU baseline only
    calls, data = cpu_sample_inputs(hot, np, stages=stages)
    smooth = np.exp(np.random.default_rng(1).uniform(-1, 1, hot.width)).astype(np.float32)
    global MOD_GAIN, MOD_SHIFT
    rng = np.random.default_rng(2)
    MOD_GAIN = (1.0 + 0.3 * rng.standard_normal((2 * hot.batch, hot.width))).astype(np.float32)
    MOD_SHIFT = (0.5 * rng.standard_normal((2 * hot.batch, hot.width))).astype(np.float32)
    nbytes = sum(c.bytes for c in calls)
    for _ in range(warmup):
        cpu_run_sample(calls, data, smooth, P)
    times = []
    t_end = time.perf_counter() + seconds
    while (steps is None and time.perf_counter() < t_end and len(times) < 50) or (steps is not None and len(times) < steps):
        t0 = time.perf_counter()
        cpu_run_sample(calls, data, smooth, P)
        times.append(time.perf_counter() - t0)
        if steps is None and len(times) >= 2 and sum(times) > seconds:
            break
    mean = sum(times) / len(times)
    return {
        "value": nbytes / mean / 1e9, "unit": UNIT, "cores": P.num_threads(), "kind": "port",
        "sample": f"1 of {hot.depth} blocks x {'all ' + str(len(hot.patch_nums)) if not stages else 'the first ' + str(stages)} stages of {hot.name} ({nbytes / 1e9:.2f} GB algorithmic, "
                  f"{len(calls)} calls), {len(times)} repeats, {mean:.3f} s each; oracle/fakequant_port.c on {P.num_threads()} threads",
    }, mean, len(times)


def reference_cpu_leg(hot, steps, warmup, budget_s, stages=0):
    """The reference's CPU implementation of the path on this box's host cores: its own torch functions from baseline/_ref
    when the reference is installed (kind "reference"), else the C port of the oracle (kind "port")."""
    from baseline import ref_env
    if ref_env.available() and not stages:
        from baseline import ref_legs
        return ref_legs.cpu_reference_sample(hot, max_rows=2048, steps=steps, warmup=warmup, budget_s=budget_s)
    return cpu_baseline(hot, 0.0, steps=steps, warmup=warmup, stages=stages)


def run_reference(args, hot):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    stages = args.sample_stages
    if stages:
        base, mean, n = cpu_baseline(hot, 0.0, steps=steps, warmup=max(1, warmup), stages=stages)
    else:
        base, mean, n = reference_cpu_leg(hot, steps, max(1, warmup), budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32/f16", "data": "synthetic",
        "config": bench_config(hot, args.gpus),
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------
class Arena:
    """A big device buffer handed out in rotating slices, so that no call re-reads bytes that could
    still sit in the 126 MB L2 from an earlier call."""

    def __init__(self, tensor):
        self.t = tensor
        self.nbytes = tensor.numel() * tensor.element_size()
        self.base = tensor.data_ptr()
        self.cur = 0

    def take(self, nbytes):
        nbytes_al = (nbytes + 255) // 256 * 256
        if nbytes_al > self.nbytes:
            raise RuntimeError("arena too small")
        if self.cur + nbytes_al > self.nbytes:
            self.cur = 0
        p = self.base + self.cur
        self.cur += nbytes_al
        return p


def synthetic_step(torch, hot, dev, rank):
    """The step's synthetic inputs, resident in HBM and the same on every run with the same workload and rank: the arenas,
    the GALT factors and adaLN tensors of the rotate sites, and the plan, (call, input pointer, output pointer) per call."""
    C = hot.width
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    GiB = 1 << 30
    a_f32 = torch.randn(GiB // 4 * 2, generator=g, device=dev, dtype=torch.float32)               # 2 GiB N(0,1) fp32
    a_f16 = torch.randn(GiB // 2, generator=g, device=dev, dtype=torch.float32).to(torch.float16)  # 1 GiB N(0,1) fp16
    a_gelu = torch.nn.functional.gelu(torch.randn(GiB, generator=g, device=dev, dtype=torch.float32), approximate="tanh").to(torch.float16)  # 2 GiB
    a_out = torch.empty(2 * GiB, dtype=torch.uint8, device=dev)
    arenas = {"f32": Arena(a_f32), "f16": Arena(a_f16), "gelu": Arena(a_gelu), "out": Arena(a_out)}
    gs = torch.Generator(device="cpu"); gs.manual_seed(7)
    smooth = {site: torch.exp(torch.rand(C, generator=gs) * 2 - 1).to(dev) for site in ("mat_qkv", "fc1")} if hot.rotate_transform else {}
    modulate = {site: (1.0 + 0.3 * torch.randn(2 * hot.batch, C, generator=gs), 0.5 * torch.randn(2 * hot.batch, C, generator=gs))
                for site in ("mat_qkv", "fc1")} if hot.modulate else {}
    modulate = {k: (a.to(dev), b.to(dev)) for k, (a, b) in modulate.items()}
    plan = [(c, in_arena(arenas, c).take(c.in_bytes), arenas["out"].take(c.out_bytes)) for c in hot.calls()]
    return arenas, smooth, modulate, plan


def in_arena(arenas, c):
    """The input arena a call reads: fp32, GELU-skewed fp16 (fc2) or N(0,1) fp16."""
    if c.in_dtype == "f32":
        return arenas["f32"]
    return arenas["gelu"] if c.site == "fc2" else arenas["f16"]


DUMP_SAMPLES = 8192     # per call: the 1200 calls of the d30 step give 39 MB of float32


def slice_intact(plan, i):
    """Whether call i's output slice still holds its output at the end of the step: no later call of the plan writes into it."""
    c, _, po = plan[i]
    return all(q + d.out_bytes <= po or q >= po + c.out_bytes for d, _, q in plan[i + 1:])


def dump_outputs(torch, np, path, plan, replay, out_arena, stream):
    """--dump-outputs: a fixed sample (seeded by the call's index) of every call's output of the step just replayed, float32,
    one [depth, samples] array per (stage, site).  The out arena is smaller than one step's output, so a later call of the
    step may have written over an earlier call's slice: a slice left intact is sampled where the step wrote it, any other
    call is launched once more on the same input into a scratch buffer (same kernel, same input bytes)."""
    os.makedirs(path, exist_ok=True)
    dev = out_arena.t.device
    n = min(DUMP_SAMPLES, min(c.elems for c, _, _ in plan))
    scratch = torch.empty(max(c.out_bytes for c, _, _ in plan), dtype=torch.uint8, device=dev)
    rows = {}
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(stream):
        for i, (c, pi, po) in enumerate(plan):
            if slice_intact(plan, i):
                out = out_arena.t[po - out_arena.base:][:c.out_bytes]
            else:
                replay.launch(c, pi, scratch.data_ptr(), stream.cuda_stream)
                out = scratch[:c.out_bytes]
            idx = torch.from_numpy(np.random.default_rng(i).integers(0, c.elems, n)).to(dev)
            vals = out.view(torch.float16 if c.out_dtype == "f16" else torch.float32)[idx].float()
            rows.setdefault((c.stage, c.site), []).append(vals.cpu().numpy())
    for (stage, site), r in rows.items():
        np.save(os.path.join(path, f"s{stage}_{site}.npy"), np.stack(r))


def config1_extra(torch, lib, dev, side):
    """BASELINE configs[0]: per-group (g=128) fp_e2 fake-quant of a synthetic fp32 4096x4096 tensor -- this library on the GPU
    (8 rotating buffer pairs = 1 GiB, so L2 cannot serve repeats) next to the CPU port of the reference's torch path
    (fp_quant_e2_per_group, argmin rule) on the same tensor."""
    import numpy as np
    from oracle import port as P
    n = 4096 * 4096
    xs = [torch.randn(4096, 4096, device=dev) for _ in range(8)]
    os_ = [torch.empty_like(t) for t in xs]
    out = {}
    for tie_name, tie in (("kernel_rule", 0), ("argmin_rule", 1)):
        with torch.cuda.stream(side):
            for i in range(8):
                lib.fpq_fake_quant(xs[i].data_ptr(), os_[i].data_ptr(), n // 128, 128, 0, 0, 0, tie, 0, side.cuda_stream)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(side)
            for i in range(64):
                lib.fpq_fake_quant(xs[i % 8].data_ptr(), os_[i % 8].data_ptr(), n // 128, 128, 0, 0, 0, tie, 0, side.cuda_stream)
            e1.record(side)
            side.synchronize()
        out[f"gpu_GBps_{tie_name}"] = 64 * n * 8 / (e0.elapsed_time(e1) / 1e3) / 1e9
    xh = xs[0].cpu().numpy()
    P.fake_quant(xh, "e2m1", 128, "argmin")
    t0 = time.perf_counter()
    for _ in range(3):
        P.fake_quant(xh, "e2m1", 128, "argmin")
    t_cpu = (time.perf_counter() - t0) / 3
    out["cpu_port_GBps_argmin_rule"] = n * 8 / t_cpu / 1e9
    out["cpu_cores"] = P.num_threads()
    out["workload"] = "fp32 4096x4096, g=128, fp_e2 (134 MB algorithmic per call)"
    return out


def generation_leg(torch, dist, dev, hot, iters, rank, world):
    """BASELINE.json's second metric: images/sec of a whole class-conditional generation pass (autoregressive pass +
    VQVAE decode) of the workload's VAR, random-init weights, with the hot path in place — `fused` = level (c) of
    INTEGRATION.md — next to the unquantized fp16 model.  The model around the hot path is tools/var_generate.py (a
    measurement harness; its GEMMs / attention / convolutions are torch library calls).  Every rank runs its own
    batches (classes sharded, no collective on the path); times are CUDA events, max over ranks."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("var_generate", os.path.join(ROOT, "tools", "var_generate.py"))
    vg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(vg)
    res = 512 if hot.patch_nums[-1] == 32 else 256
    bits = 6 if hot.act_fmt in ("e2m3", "e3m2") else 4
    out = {"unit": "images/s", "model": f"VAR-d{hot.depth} {res}x{res}, B={hot.batch}/GPU, W{bits}A{bits}, random init",
           "harness": "tools/var_generate.py", "iters": iters, "warmup": 1}
    for mode in (("fused" if hot.rotate_transform else "modules"), "fp16"):
        ms, err = float("nan"), None
        try:
            r = vg.measure(dev, hot.depth, hot.batch, res, bits, mode, iters, 1, rank, world, rotate=hot.rotate_transform)
            ms = r["ms_per_batch"]
            if not r["finite"]:
                err = "non-finite image"
        except Exception as e:  # noqa: BLE001  (reported in the JSON line; the hot-path numbers above stand on their own)
            err = f"{type(e).__name__}: {e}"
        t = torch.tensor([ms if err is None else float("inf")], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        worst = float(t.item())
        if worst == float("inf"):
            out[mode] = {"error": err or "failed on another rank"}
        else:
            out[mode] = {"images_per_sec": world * hot.batch / (worst / 1e3), "ms_per_batch": worst,
                         "decode_ms_per_batch": r["decode_ms_per_batch"], "fpq_launches_per_batch": r["fpq_launches_per_batch"]}
    return out


def ncu_traffic(dom_key, bytes_per_avg_launch):
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed
    `ncu --set full` capture (profiles/r2_traffic.json, written by tools/ncu_summary.py from the .ncu-rep), scaled from the
    captured launch to the step's average launch by algorithmic bytes (traffic / algorithmic is what the capture measures)."""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        table = json.load(f)
    op, fmt, din, dout = dom_key
    ent = table.get(f"{op}:{fmt}:{din}->{dout}")
    if not ent:
        return None
    ratio = ent["dram_bytes"] / ent["algorithmic_bytes"]
    return {"per_avg_launch": ratio * bytes_per_avg_launch, "captured_launch": ent, "ratio_dram_over_algorithmic": ratio}


def reference_gpu_legs(torch, dev, hot, args):
    """(reference_gpu_path, generation_reference_model): the UNMODIFIED reference from baseline/_ref on this GPU, each in a
    child process (the reference's code owns that process: it switches torch's initialisers off, and a device-side assert
    in it cannot take this run down)."""
    from baseline import ref_env
    if not ref_env.available():
        why = {"unavailable": ref_env.why_unavailable()}
        return why, why

    def child(cmd, timeout):
        r = subprocess.run([sys.executable] + cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
        lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
        if r.returncode != 0 and not lines:
            raise RuntimeError((r.stderr.strip().splitlines() or ["exit code %d" % r.returncode])[-1][:300])
        return lines

    try:
        gpu = child(["-m", "baseline.ref_legs", "gpu_step", hot.name], 600)[-1]
    except Exception as e:  # noqa: BLE001  (reported in the JSON line)
        gpu = {"error": f"{type(e).__name__}: {e}"}
    gen = None
    if not args.no_generation and hot.rotate_transform:
        res = 512 if hot.patch_nums[-1] == 32 else 256
        bits = 6 if hot.act_fmt in ("e2m3", "e3m2") else 4
        gen = {"unit": "images/s", "model": f"the reference's own VAR-d{hot.depth} {res}x{res} (build_vae_var, autoregressive_infer_cfg, fp16 autocast), "
                                             f"B={hot.batch}, W{bits}A{bits}, random init", "harness": "tools/ref_model_generate.py"}
        for mode in ("fp16", "reference", "dropin", "fused"):
            try:
                r = child([os.path.join(ROOT, "tools", "ref_model_generate.py"), "--depth", str(hot.depth), "--batch", str(hot.batch), "--res", str(res),
                           "--bits", str(bits), "--iters", "2", "--modes", mode], 900)[-1]
                gen[mode] = {k: r[k] for k in ("images_per_sec", "ms_per_batch", "finite", "fpq_launches_per_batch")}
                gen["galt_factors"] = r["galt_factors"]
            except Exception as e:  # noqa: BLE001
                gen[mode] = {"error": f"{type(e).__name__}: {e}"}
    return gpu, gen


def other_configs(args):
    """BASELINE configs[1] and [3] (VAR-d16 plain, VAR-d36 W6A6 rotate): the device-resident step of each, measured by a
    short child run of this script (its own process: fresh arenas, same timing code)."""
    out = {}
    for wl in ("var_d16_w4a4", "var_d36_w6a6_rot"):
        if wl == args.workload:
            continue
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--workload", wl, "--steps", "10", "--warmup", "3", "--no-e2e", "--no-cpu",
                                "--no-generation", "--no-reference-legs", "--no-other-configs", "--no-search"], capture_output=True, text=True, timeout=300)
            d = json.loads(r.stdout.strip().splitlines()[-1])
            out[wl] = {"value": d["value"], "unit": d["unit"], "ms_per_step": d["ms_per_step"], "frac_of_measured_peak": d["value"] / d["roofline"]["peak"],
                       "desc": d["config"]["desc"], "kernels": {k: v["GB/s"] for k, v in d["kernels"].items()}}
        except Exception as e:  # noqa: BLE001
            out[wl] = {"error": f"{type(e).__name__}: {e}"}
    return out


def search_leg(torch, dist, dev, rank, world, blocks, depth=30, acts=1000):
    """BASELINE configs[4] (FP4 format search, search/search_fp4_format.py:781-836) on a BOUNDED unit list: the four layers
    of `blocks` VAR-d30 blocks (the full sweep has 30), random-init weights, the reference's calibration shapes (per layer 1000
    tensors [2, pn^2, C_in] = 136 000 rows; N(0,1), GELU-skewed for fc2), candidates {e1m2, e2m1, e3m0} x {e1m2, e2m1, e3m0}.
    (layer, weight-format) units are dealt round-robin to the ranks (strong scaling: the unit list does not grow with N),
    every rank scores its units with fpqvar_b200.search.search_layer_batched (fused quantizers, library GEMMs, fused
    squared-error reduction) and ONE all-reduce of the [layers, 3, 3] float64 table ends the sweep.  CUDA events, max over ranks."""
    from fpqvar_b200 import search
    C = 64 * depth
    patch = (1, 2, 3, 4, 5, 6, 8, 10, 13, 16)
    rows = [2 * patch[j % 10] ** 2 for j in range(acts)]
    shapes = {"mat_qkv": (3 * C, C, torch.float32, False), "proj": (C, C, torch.float16, False),
              "fc1": (4 * C, C, torch.float32, False), "fc2": (C, 4 * C, torch.float16, True)}
    names = [(b, n) for b in range(blocks) for n in shapes]
    units = [(li, wi) for li in range(len(names)) for wi in range(len(search.FP4_FORMATS))]
    mine = [units[u] for u in range(rank, len(units), world)]
    table = torch.zeros(len(names), 3, 3, dtype=torch.float64, device=dev)

    def layer(li):
        b, n = names[li]
        o, i, dt, gelu = shapes[n]
        g = torch.Generator(device=dev).manual_seed(1000 * b + list(shapes).index(n))       # the same data on whichever rank owns the unit
        w = (torch.randn(o, i, device=dev, generator=g) * 0.02).to(dt)
        x = torch.randn(sum(rows), i, device=dev, generator=g)
        if gelu:
            x = torch.nn.functional.gelu(x, approximate="tanh")
        return w, list(x.to(dt).split(rows))

    def run(scorer=None):
        scorer = scorer or search.search_layer_batched
        table.zero_()
        cur, data = None, None
        for li, wi in mine:
            if li != cur:
                cur, data = li, layer(li)
            table[li, wi] = scorer(data[0], data[1], [search.FP4_FORMATS[wi]], search.FP4_FORMATS)[0]
        if world > 1:
            dist.all_reduce(table)

    def timed(scorer):
        run(scorer)                                 # warm-up (cuBLAS heuristics, allocator)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(scorer)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / 1e3], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # the reference's search scripts never enable TF32: the fp32 GEMMs of the mat_qkv / fc1 layers run at full precision
    # (the generation harness above switches TF32 on, like evaluate_fp_quant_transform_rotate.py:171-175 -- undo that here)
    tf32_saved = (torch.backends.cuda.matmul.allow_tf32, torch.get_float32_matmul_precision())
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")
    # the same sweep with the candidates evaluated from codes on the tensor cores and the loss taken in the GEMM's epilogue
    # (search.search_layer_lowbit, SURVEY section 8 f3); then the fake-quant + library-GEMM path, whose table is the one reported
    secs_lowbit = timed(search.search_layer_lowbit)
    table_lowbit = table.clone()
    secs = timed(None)
    torch.backends.cuda.matmul.allow_tf32 = tf32_saved[0]
    torch.set_float32_matmul_precision(tf32_saved[1])
    best = [search.best_formats(table[li], search.FP4_FORMATS, search.FP4_FORMATS) for li in range(len(names))]
    best_lb = [search.best_formats(table_lowbit[li], search.FP4_FORMATS, search.FP4_FORMATS) for li in range(len(names))]
    rel = float(((table_lowbit - table).abs() / table.abs().clamp_min(1e-300)).max().item())
    lowbit = {"seconds": secs_lowbit, "units_per_sec": len(units) / secs_lowbit, "max_rel_diff_of_loss_table": rel,
              "same_winners": all(a["weight_format"] == b["weight_format"] and a["activation_format"] == b["activation_format"]
                                  for a, b in zip(best, best_lb)),
              "what": "search_layer_lowbit: quantizers emit codes, tcgen05 e4m3-container GEMM, loss in the epilogue (nothing written)"}
    return {"seconds": secs, "lowbit": lowbit, "units": len(units), "units_per_sec": len(units) / secs, "layers": len(names), "scaling": "strong",
            "calibration_rows_per_layer": sum(rows), "activations_per_layer": acts,
            "desc": f"FP4 format search, {blocks} of {depth} VAR-d30 blocks x 4 layers x 3 weight formats = {len(units)} units over {world} rank(s); "
                    "per unit: 3 activation formats, output-level loss over 1000 row-stacked calibration tensors",
            "winners": {f"blocks.{b}.{n}": f"w={best[i]['weight_format']},a={best[i]['activation_format']}" for i, (b, n) in enumerate(names)}}


def lowbit_gemm_leg(torch, dev, peaks):
    """SURVEY.md section 8 f4: the four linears of one VAR-d30 block at the largest stage (25 600 token rows) as REAL low-bit GEMMs
    from packed codes (fpqvar_b200.lowbit: tcgen05.mma kind::f8f6f4 on e4m3 containers) beside what the reference runs -- the
    fp16 library GEMM on the fake-quantized tensors (QuantizedLinear.forward, qu.py:764-769).  `group128` = one scale per (row,
    128-group) on both operands (the README W4A4 configuration; bit-exact against oracle/gemm_codes.c), `row` = per_token x
    per_channel (the README W6A6 configuration).  CUDA events, 20 launches after 3 warm-ups, outputs rotate through 4 buffers."""
    from fpqvar_b200 import lowbit, ops
    C, rows = 1920, 25600
    layers = {"mat_qkv": (3 * C, C), "proj": (C, C), "fc1": (4 * C, C), "fc2": (C, 4 * C)}

    def timeit(fn, iters=20, warm=3):
        for i in range(warm):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters / 1e3

    out, tot = {}, {"group128": 0.0, "row": 0.0, "fp16_library": 0.0, "flop": 0.0}
    g = torch.Generator(device=dev).manual_seed(7)
    for name, (n, k) in layers.items():
        x = torch.randn(rows, k, device=dev, dtype=torch.float16, generator=g)
        w = torch.randn(n, k, device=dev, generator=g) * 0.02
        outs = [torch.empty(rows, n, device=dev, dtype=torch.float16) for _ in range(4)]
        a, ww = lowbit.pack_codes(x, "e2m1"), lowbit.pack_codes(w, "e2m1")
        ar, wr = lowbit.pack_codes(x, "e2m1", True), lowbit.pack_codes(w, "e2m1", True)
        xq, wq = ops.fake_quant(x, "e2m1", 128, "kernel"), ops.fake_quant(w, "e2m1", 128, "kernel").half()
        flop = 2.0 * rows * n * k
        t_g = timeit(lambda i: lowbit.linear_codes(a, ww, None, torch.float16, outs[i % 4]))
        t_r = timeit(lambda i: lowbit.linear_codes(ar, wr, None, torch.float16, outs[i % 4]))
        t_l = timeit(lambda i: torch.nn.functional.linear(xq, wq))
        t_p = timeit(lambda i: lowbit.pack_codes(x, "e2m1"))
        t_f = timeit(lambda i: ops.fake_quant(x, "e2m1", 128, "kernel"))
        out[name] = {"m_n_k": [rows, n, k], "group128_TFLOPs": flop / t_g / 1e12, "row_TFLOPs": flop / t_r / 1e12,
                     "fp16_library_on_fake_quantized_TFLOPs": flop / t_l / 1e12,
                     "quantize_to_codes_us": t_p * 1e6, "quantize_to_codes_GBps": rows * k * 3.03 / t_p / 1e9, "fake_quant_us": t_f * 1e6}
        for key, t in (("group128", t_g), ("row", t_r), ("fp16_library", t_l)):
            tot[key] += t
        tot["flop"] += flop
        del x, w, outs, a, ww, ar, wr, xq, wq
    peak = peaks.get("bf16_tflops") if peaks else None
    return {"layers": out,
            "block_TFLOPs": {k: tot["flop"] / tot[k] / 1e12 for k in ("group128", "row", "fp16_library")},
            "roofline": {"bound": "tensor", "kernel": "gemm_codes_kernel<256, 128> (row scales)", "achieved": tot["flop"] / tot["row"] / 1e12,
                         "peak": 2 * peak if peak else None, "unit": "TFLOP/s",
                         "frac": tot["flop"] / tot["row"] / 1e12 / (2 * peak) if peak else None,
                         "peak_source": "2 x MEASURED_PEAKS.json bf16_tflops (the 8-bit tensor rate is twice the 16-bit one; no measured 8-bit figure on this pool)"},
            "what": "VAR-d30 block at the largest stage, W4A4 e2m1 x e2m1 from codes; see profiles/r2_gemm_codes.txt for the variants"}


def main():
    args = parse_args()
    from fpqvar_b200.var_workload import WORKLOADS
    hot = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, hot)
        return

    import torch
    import torch.distributed as dist
    from fpqvar_b200 import _lib as L
    from fpqvar_b200.hotpath import DeviceReplay, HostPipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.lib()

    calls = hot.calls()
    step_bytes = sum(c.bytes for c in calls)
    in_bytes = sum(c.in_bytes for c in calls)
    out_bytes = sum(c.out_bytes for c in calls)

    arenas, smooth, modulate, plan = synthetic_step(torch, hot, dev, rank)
    replay = DeviceReplay(dev, smooth, modulate=modulate)

    def issue(subset, stream):
        for c, pi, po in subset:
            replay.launch(c, pi, po, stream)

    side = torch.cuda.Stream(dev)

    def capture(subset):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            issue(subset[:8], side.cuda_stream)           # make sure lazy init happened outside capture
            side.synchronize()
            n0 = lib.fpq_launch_count()
            with torch.cuda.graph(gr, stream=side):
                issue(subset, side.cuda_stream)
            n_launch = lib.fpq_launch_count() - n0
        return gr, int(n_launch)

    graph, launches_per_step = capture(plan)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_replays(gr, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with torch.cuda.stream(side):
            e0.record(side)
            for _ in range(k):
                gr.replay()
            e1.record(side)
        barrier()
        return e0.elapsed_time(e1) / 1e3

    n_warm = 1 if args.profile else max(3, args.warmup)
    for _ in range(n_warm):
        graph.replay()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_dev = timed_replays(graph, args.steps)
    if args.dump_outputs and rank == 0:
        import numpy as np
        dump_outputs(torch, np, args.dump_outputs, plan, replay, arenas["out"], side)
    if args.profile:
        if sampler:
            sampler.stop()
        if rank == 0:
            print(json.dumps({"profile_run": True, "steps": args.steps, "launches_per_step": launches_per_step,
                              "value_under_profiler_is_not_a_bench_value": world * args.steps * step_bytes / t_dev / 1e9}))
        return

    # ---- roofline of the dominant kernel (timed alone, same inputs) --------------------------
    by_kernel = {}
    for item in plan:
        c = item[0]
        by_kernel.setdefault((c.op, c.fmt, c.in_dtype, c.out_dtype), []).append(item)
    dom_key = max(by_kernel, key=lambda k: sum(i[0].bytes for i in by_kernel[k]))
    fam = {}
    for key, items in by_kernel.items():
        gr, n_l = capture(items)
        for _ in range(3):
            gr.replay()
        fam[key] = (timed_replays(gr, args.steps), n_l, sum(i[0].bytes for i in items))
    t_dom, dom_launches, dom_bytes = fam[dom_key]
    dom = by_kernel[dom_key]
    # the big-stage launches of that kernel alone (bandwidth-bound regime; the early stages are launch-latency-bound)
    big = [i for i in dom if i[0].bytes >= 64 << 20]
    big_graph, _ = capture(big)
    for _ in range(3):
        big_graph.replay()
    t_big = timed_replays(big_graph, args.steps)
    big_bytes = sum(i[0].bytes for i in big)
    clocks = sampler.stop() if sampler else None

    # ---- e2e: host buffers through HostPipeline ----------------------------------------------
    e2e = None
    if not args.no_e2e:
        from fpqvar_b200.hotpath import bind_to_gpu_numa
        numa_cpus = bind_to_gpu_numa(local_rank)          # before the pinned buffers exist: first touch places them on the GPU's node
        max_in = max(c.in_bytes for c in calls)
        max_out = max(c.out_bytes for c in calls)
        pipe = HostPipeline(dev, max_in, max_out, smooth, modulate=modulate, slots=3)
        h_f32 = torch.randn(max(c.in_bytes for c in calls if c.in_dtype == "f32") // 4 if any(c.in_dtype == "f32" for c in calls) else 1).pin_memory()
        h_f16 = torch.nn.functional.gelu(torch.randn(max(c.in_bytes for c in calls if c.in_dtype == "f16") // 2), approximate="tanh").to(torch.float16).pin_memory()
        h_out = [torch.empty(max_out, dtype=torch.uint8).pin_memory() for _ in range(3)]
        v32, v16 = h_f32.view(torch.uint8), h_f16.view(torch.uint8)
        hin = [v32 if c.in_dtype == "f32" else v16 for c in calls]
        hout = [h_out[i % 3] for i in range(len(calls))]
        pipe.run(calls[: 4 * hot.depth], hin, hout)        # warm-up: the first stage
        pipe.synchronize()
        n_e2e = max(1, args.e2e_steps)
        barrier()
        t0 = time.perf_counter()
        n0 = lib.fpq_launch_count()
        for _ in range(n_e2e):
            pipe.run(calls, hin, hout)
        pipe.synchronize()
        barrier()
        t_e2e = time.perf_counter() - t0
        e2e_launches = int(lib.fpq_launch_count() - n0)
        if world > 1:
            t = torch.tensor([t_e2e], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_e2e = float(t.item())
        e2e = {"value": world * n_e2e * step_bytes / t_e2e / 1e9, "unit": UNIT, "h2d_bytes_per_step": world * in_bytes,
               "d2h_bytes_per_step": world * out_bytes, "steps": n_e2e, "ms_per_step": t_e2e / n_e2e * 1e3,
               "api": "fpqvar_b200.hotpath.HostPipeline.run (pinned host buffers -> C ABI -> pinned host buffers)",
               "launches": e2e_launches, "host_binding": f"rank bound to its GPU's NUMA node (cpus {numa_cpus})" if numa_cpus else "no NUMA information: unbound",
               "staging_slots": 3}
        del pipe

    # ---- images/sec: the caller around the hot path (SURVEY.md section 8d) --------------------
    generation = None
    if not args.no_generation:
        generation = generation_leg(torch, dist, dev, hot, args.gen_iters, rank, world)

    # ---- format search (BASELINE configs[4]) on a bounded unit list, sharded over the ranks -------------------------
    search_res = None
    if not args.no_search and hot.depth == 30:
        try:
            search_res = search_leg(torch, dist, dev, rank, world, args.search_blocks)
        except Exception as e:  # noqa: BLE001
            search_res = {"error": f"{type(e).__name__}: {e}"}

    # ---- real low-bit GEMMs from codes beside the fp16 library GEMM on the fake-quantized tensors (SURVEY section 8 f4; rank 0) ----
    lowbit_res = None
    if rank == 0 and not args.no_lowbit:
        try:
            mp = os.path.join(ROOT, "MEASURED_PEAKS.json")
            lowbit_res = lowbit_gemm_leg(torch, dev, json.load(open(mp)) if os.path.exists(mp) else None)
        except Exception as e:  # noqa: BLE001
            lowbit_res = {"error": f"{type(e).__name__}: {e}"}
    if world > 1:
        dist.barrier()

    # ---- the reference's own GPU path and its own model on this box (rank 0, N=1; outside every timed region above) ----
    reference_gpu = generation_ref = other = None
    if world == 1 and not args.no_reference_legs:
        del replay, graph, big_graph, arenas, plan
        torch.cuda.empty_cache()
        reference_gpu, generation_ref = reference_gpu_legs(torch, dev, hot, args)
    if world == 1 and not args.no_other_configs:
        other = other_configs(args)

    # ---- gather (the only collective) --------------------------------------------------------
    if world > 1:
        keys = sorted(fam)
        t = torch.tensor([t_dev, t_dom, t_big] + [fam[k][0] for k in keys], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        vals = [float(v) for v in t.tolist()]
        t_dev, t_dom, t_big = vals[:3]
        fam = {k: (vals[3 + i], fam[k][1], fam[k][2]) for i, k in enumerate(keys)}

    if rank == 0:
        peak, peak_src = load_peaks()
        value = world * args.steps * step_bytes / t_dev / 1e9
        dom_gbs = args.steps * dom_bytes / t_dom / 1e9
        big_gbs = args.steps * big_bytes / t_big / 1e9
        def kernel_name(key):
            op, fmt, din, dout = key
            if op == "rotate_quant":
                return f"transform_rotate_quant_{{stream,small}}_kernel<{fmt}> (f32->f16)"
            if op == "mod_rotate_quant":
                return f"modulate_transform_rotate_quant_{{stream,small}}_kernel<{fmt}> (adaLN modulate fused, f32->f16)"
            packed = din == "f16" and dout == "f16"
            base = {"group": "fake_quant_group", "signsplit": "signsplit_group"}[op]
            return f"{base}_h16_kernel<{fmt}> (f16->f16)" if packed else f"{base}_kernel<{din}->{dout},{fmt}>"
        kname = kernel_name(dom_key)
        traffic = ncu_traffic(dom_key, dom_bytes / max(1, dom_launches))
        kernels = {kernel_name(k): {"GB/s": args.steps * b / t / 1e9, "launches_per_step": n_l, "share_of_step_bytes": b / step_bytes,
                                    "ms_per_step_alone": t / args.steps * 1e3} for k, (t, n_l, b) in fam.items()}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": n_warm,
            "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32/f16", "data": "synthetic",
            "config": bench_config(hot, world),
            "roofline": {
                "bound": "hbm", "kernel": kname, "achieved": dom_gbs, "peak": peak,
                "unit": "GB/s", "frac": dom_gbs / peak, "traffic": traffic["per_avg_launch"] if traffic else None, "peak_source": peak_src,
                "launches_per_step": dom_launches, "avg_launch_us": t_dom / args.steps / max(1, dom_launches) * 1e6,
                "bytes_per_launch": dom_bytes / max(1, dom_launches),
                "large_launches": {"min_bytes": 64 << 20, "achieved": big_gbs, "frac": big_gbs / peak, "n": len(big)},
                "frac_of_nominal_8TBps": dom_gbs / 8000.0,
                "traffic_detail": traffic,
            },
            "kernels": kernels,
            "images_per_sec_hot_path_only": world * hot.batch / (t_dev / args.steps),
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
        }
        if e2e is not None:
            line["e2e"] = e2e
        if generation is not None:
            line["generation"] = generation
        if search_res is not None:
            line["search"] = search_res
        if lowbit_res is not None:
            line["lowbit_gemm"] = lowbit_res
        if reference_gpu is not None:
            line["reference_gpu_path"] = reference_gpu
        if generation_ref is not None:
            line["generation_reference_model"] = generation_ref
        if other is not None:
            line["other_configs"] = other
        if world == 1 and not args.no_cpu:
            base, _, _ = reference_cpu_leg(hot, 1, 1, budget_s=2 * args.cpu_seconds)
            line["cpu_baseline"] = base
            if base["kind"] != "port":
                port, _, _ = cpu_baseline(hot, args.cpu_seconds)
                line["cpu_port"] = port
            line["config1"] = config1_extra(torch, lib, dev, side)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
