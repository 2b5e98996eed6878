#!/usr/bin/env python
"""bench.py -- tokens/sec of the LSTM-LM train step (main.py:109-117) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config large|medium|small]
                    [--impl ours|reference] [--engine tc|simt] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over one synthetic
[T,B] window per GPU: forward, softmax-NLL, backward, (gradient all-reduce when N>1),
global-norm clip, SGD.  Weak scaling: B=20 per GPU, rows of the global batch are
independent token streams (main.py:63-66), so no data-path collective except the one
gradient all-reduce.

  value      whole-job tokens/s, tokens already resident in HBM, CUDA events, max over ranks
  e2e        same step through the public host-buffer call (`Trainer.train_step_host` ->
             zrb_train_step_host): CPU [T,B] int64 views as main.py:71-72 builds them, H2D of
             x,y and D2H of the loss inside the timed region
  roofline   dominant kernel class, timed live with CUDA events on the launching stream in a
             second instrumented pass of the same K steps (zrb_prof_*)
  cpu_baseline  oracle/torch_port.py (the reference's own torch calls) on the host cores
  --impl reference   that CPU port alone, same config / metric (rank 0 only)
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

CONFIGS = {
    # name: V, H, L, T, B, dropout, winit, lr, max_norm   (README.md:20-27 recipes)
    "small": dict(V=10000, H=200, L=2, T=20, B=20, p=0.0, winit=0.1, lr=1.0, clip=5.0),
    "medium": dict(V=10000, H=650, L=2, T=35, B=20, p=0.5, winit=0.05, lr=1.0, clip=5.0),
    "large": dict(V=10000, H=1500, L=2, T=35, B=20, p=0.65, winit=0.04, lr=1.0, clip=10.0),
}
METRIC = "tokens/sec (and valid perplexity) Large-LSTM 1500h at 1/2/4/8 B200 vs ref CPU"


def workload_name(name, c):
    return (f"{name}: {c['L']}x{c['H']} LSTM LM train step, T={c['T']}, B={c['B']}/GPU, V={c['V']}, "
            f"dropout {c['p']}, synthetic uniform tokens")


def flops_per_token(c):
    """SURVEY 8d: train FLOPs/token = 3 * (16*L*H^2 + 2*H*V)."""
    return 3 * (16 * c["L"] * c["H"] ** 2 + 2 * c["H"] * c["V"])


def clip_sgd_bytes(c, fused):
    """Bytes the optimiser class has to move (DESIGN.md 4.4).  fused = the single-process `Trainer` step: the
    matrices' sum of squares comes from the wgrad GEMM epilogues, coef*g is not stored back, only the window's
    embedding rows are touched -> per matrix element 4 (g) + 4 + 4 (p read, write) + fp16 images; otherwise
    (data parallel / keep_clipped_grads) the reference's passes: norm read 4 B + g read/write 8 B + p 8 B."""
    N, H, L, V = c["T"] * c["B"], c["H"], c["L"], c["V"]
    mats = L * 8 * H * H + V * H                       # w_ih, w_hh per layer + fc.W
    small = L * 8 * H + V                              # biases
    images = (L * 4 * H * H) * 2 + (L * 4 * H * H) * 4 + V * H * 2    # w_ih rows, w_hh fwd+bwd slices, fc rows
    if fused:
        return mats * 12 + images + small * 16 + N * H * 16
    return (mats + V * H + small) * 20 + images


def class_work(c, fused_update=True):
    """Algorithmic work of one step per kernel class: (kind, amount) with FLOPs for the dense
    contractions and bytes for the streaming kernels (DESIGN.md section 'Kernels')."""
    N, H, L, V = c["T"] * c["B"], c["H"], c["L"], c["V"]
    P = 2 * V * H + V + L * (8 * H * H + 8 * H)
    return {
        "gemm_in": ("flop", 8 * N * H * H * L), "rec_fwd": ("flop", 8 * N * H * H * L),
        "proj_fwd": ("flop", 2 * N * H * V), "proj_bwd": ("flop", 4 * N * H * V),
        "rec_bwd": ("flop", 8 * N * H * H * L), "gemm_dx": ("flop", 8 * N * H * H * L),
        "gemm_wgrad": ("flop", 16 * N * H * H * L),
        "softmax": ("byte", N * V * 4 + N * V * 2), "clip_sgd": ("byte", clip_sgd_bytes(c, fused_update)),
        "embed_fwd": ("byte", 2 * N * H * 4), "embed_bwd": ("byte", V * H * 4 + 2 * N * H * 4),
        "pack": ("byte", 6 * (P - V * H - V)),
    }


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tensor=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tensor=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([f.strip() for f in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 8 and r[4 + i].lower().startswith("active")
                                                         for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_threads():
    """torch's own default on an SMT box: half the logical CPUs (one per physical core)."""
    n = os.cpu_count() or 2
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    return max(1, n // 2)


def bench_config(name, c, world, engine, transport, device, update="end of step"):
    """`config` object shared by both arms (same keys, so the driver can compare them)."""
    return {"workload": workload_name(name, c), "device": device, "engine": engine, "parallelism": f"dp{world}",
            "weight_update": update,
            "dp_transport": transport, "global_batch": c["B"] * world, "seq_len": c["T"],
            "l2": "no flush: per-step working set (fp32 params+grads 528 MB + activations) exceeds the 126 MB L2"
            if name == "large" else "no flush; working set may fit L2 for this config"}


def gpu_baseline_leg(c, steps=40, warmup=10):
    """The bar BASELINE.json's north_star names: the reference's `--lstm_type pytorch` train step on the SAME GPU
    (oracle/torch_port.py on cuda = the reference's own torch calls: cuDNN nn.LSTM, cuBLAS addmm, eager softmax,
    clip_grad_norm_, per-parameter SGD; torch default flags), CUDA-event timed, tokens handed over as CPU views
    like main.py:111 does."""
    import torch
    from oracle import torch_port as P
    model = P.TorchLstmLm(c["V"], c["H"], c["L"], c["p"], c["winit"], seed=1).cuda()
    model.train()
    data = P.synthetic_batches(c["V"], c["B"], c["T"], steps + warmup)
    states = model.zero_state(c["B"])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i, (x, y) in enumerate(data):
        if i == warmup:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record()
        _, _, states = P.train_step(model, x.cuda(), y.cuda(), states, c["lr"], c["clip"])
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps * 1e3
    ms = e0.elapsed_time(e1) / steps
    del model
    torch.cuda.empty_cache()
    return {"value": c["T"] * c["B"] / (ms * 1e-3), "unit": "tokens/s", "ms_per_step": ms, "ms_per_step_wall": wall,
            "steps": steps, "warmup": warmup, "n_gpus": 1,
            "what": "reference --lstm_type pytorch path (cuDNN nn.LSTM + cuBLAS + eager loss/clip/SGD) on this GPU, "
                    f"torch {torch.__version__}, cuDNN {torch.backends.cudnn.version()}, "
                    f"cudnn.allow_tf32={torch.backends.cudnn.allow_tf32}, matmul tf32={torch.backends.cuda.matmul.allow_tf32}"}


def cpu_port_leg(c, budget_s, steps=None, warmup=1):
    """The reference's CPU path (torch port) on the host cores; bounded sample."""
    import torch
    from oracle import torch_port as P
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the reference's CPU path (`main.py --device cpu`) uses torch's
    # default = one thread per physical core, so pin that here and the arm means the same thing at every N
    torch.set_num_threads(cpu_threads())
    if steps is None:
        dt1, _, thr = P.time_cpu_train_steps(c["V"], c["H"], c["L"], c["B"], c["T"], c["p"], c["winit"], c["lr"],
                                             c["clip"], steps=1, warmup=1)
        steps = max(3, min(200, int(budget_s / max(dt1, 1e-3))))
    dt, tps, thr = P.time_cpu_train_steps(c["V"], c["H"], c["L"], c["B"], c["T"], c["p"], c["winit"], c["lr"],
                                          c["clip"], steps=steps, warmup=warmup)
    return {"value": tps, "unit": "tokens/s", "cores": thr, "kind": "port",
            "sample": f"{steps} train steps of the same config ({steps * c['T'] * c['B']} tokens) after {warmup} "
                      f"warm-up, torch {torch.__version__} CPU (oneDNN nn.LSTM), {dt * 1e3:.1f} ms/step",
            "host_cpus": os.cpu_count()}, dt


DUMP_SAMPLE = 1 << 20       # elements kept of a larger parameter tensor: the Large config dumps ~25 MB


def dump_outputs(out_dir, tr):
    """Write what the last train step handed its caller as float32 .npy files: loss, clip norm, the carried (h, c)
    states and the updated parameters.  A parameter tensor of more than DUMP_SAMPLE elements is cut to a sample at
    fixed, seeded positions, the same in every run of the same config, so two builds compare element for element.
    Compare over few steps: fp32 atomics add in another order from run to run and the carried states amplify that
    (two runs of one build, Large, B200 at 1000 W: 2e-4 of a tensor's scale at --steps 1, 1e-3 at 10, 0.2 at 50)."""
    import numpy as np
    arrays = {"loss": tr.loss, "norm": tr.norm}
    for l, (h, c) in enumerate(tr.states):
        arrays[f"state_h{l}"], arrays[f"state_c{l}"] = h, c
    for k, p in tr.model.named_parameters():
        arrays["param_" + k] = p
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        total += a.nbytes
    assert total <= 64 << 20, total


def run_reference(args, c, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base, dt = cpu_port_leg(c, 0, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(name, c, max(1, args.gpus), "torch CPU (oneDNN)", None, "host CPU"),
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def run_ours(args, c, name):
    import torch
    import torch.distributed as dist
    import zaremba_b200
    from zaremba_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: zaremba_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    V, H, L, T, B = c["V"], c["H"], c["L"], c["T"], c["B"]
    K, W = args.steps, args.warmup
    torch.manual_seed(1)                       # same weights on every rank (replicated parameters)
    model = zaremba_b200.Model(V, H, L, c["p"], c["winit"], engine=args.engine).to(dev)
    model.train()
    tr = zaremba_b200.Trainer(model, B, T, lazy_update=not args.strict_update)
    # synthetic PTB-shaped tokens: the global batch is [B*world, .]; this rank owns rows rank*B .. rank*B+B-1
    g = torch.Generator().manual_seed(2)
    n_win = K + W
    data = torch.randint(0, V, (B * world, T * n_win + 1), generator=g, dtype=torch.int64)[rank * B:(rank + 1) * B]
    host_batches = [(data[:, i * T:(i + 1) * T].t(), data[:, i * T + 1:(i + 1) * T + 1].t()) for i in range(n_win)]
    dev_batches = [(x.contiguous().to(dev), y.contiguous().to(dev)) for x, y in host_batches]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_region(fn, batches):
        for x, y in batches[:W]:
            fn(x, y)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.zrb_launch_count()
        t0 = time.perf_counter()
        e0.record()
        for x, y in batches[W:W + K]:
            fn(x, y)
        tr.flush()            # lazy update: the last step's deferred weight updates belong to the timed region
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = torch.tensor([e0.elapsed_time(e1), wall * 1e3], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms[0].item(), ms[1].item(), lib.zrb_launch_count() - n0

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    # 1) device-resident tokens: the headline `value`
    dev_ms, _, launches = timed_region(lambda x, y: tr.train_step(x, y, c["lr"], c["clip"]), dev_batches)
    clocks = sampler.stop() if sampler else None
    loss_after = tr.loss.item()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tr)
    # replica check: after the timed steps every rank must hold bit-identical parameters (same all-reduced
    # gradients, same clip, same update) -- MAX - MIN over ranks of two checksums, must be 0
    dp_check = None
    if world > 1:
        bits = tr.flat_p.view(torch.int32).to(torch.int64)
        chk = torch.stack([bits.sum(), (bits * (torch.arange(bits.numel(), device=dev) % 8191 + 1)).sum()])
        hi, lo = chk.clone(), chk.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dp_check = {"param_checksum_max_minus_min": [int(v) for v in (hi - lo).tolist()],
                    "replicas_identical": bool((hi == lo).all().item()), "after_steps": K + W}
    # the same step in the mode that leaves coef * g in .grad like clip_grad_norm_ (main.py:115) does
    was_keep = tr._keep_clipped
    tr._keep_clipped = True                      # (also arms the copy-engine transport's wait for the peers' pulls)
    _lib.check(lib.zrb_set_keep_clipped_grads(tr.ctx, 1))
    keep_ms, _, _ = timed_region(lambda x, y: tr.train_step(x, y, c["lr"], c["clip"]), dev_batches)
    tr._keep_clipped = was_keep
    _lib.check(lib.zrb_set_keep_clipped_grads(tr.ctx, 1 if was_keep else 0))
    # 2) end to end through the host-buffer call (wall clock: H2D, step, D2H of the loss each step)
    tr.reset_states()
    _, e2e_wall_ms, _ = timed_region(lambda x, y: tr.train_step_host(x, y, c["lr"], c["clip"]), host_batches)
    # 3) instrumented pass for the per-class roofline
    import ctypes as C
    tr.reset_states()
    _lib.check(lib.zrb_prof_enable(tr.ctx, 1))
    for x, y in dev_batches[W:W + K]:
        tr.train_step(x, y, c["lr"], c["clip"])
    ms_arr = (C.c_float * len(_lib.PROF_CLASSES))()
    cnt_arr = (C.c_int64 * len(_lib.PROF_CLASSES))()
    _lib.check(lib.zrb_prof_read(tr.ctx, ms_arr, cnt_arr))
    _lib.check(lib.zrb_prof_enable(tr.ctx, 0))
    per_class = {n: (ms_arr[i] / K, cnt_arr[i] / K) for i, n in enumerate(_lib.PROF_CLASSES) if cnt_arr[i]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    tokens = T * B * world * K
    peaks = measured_peaks()
    work = class_work(c, fused_update=(world == 1))
    top = max(per_class, key=lambda n: per_class[n][0]) if per_class else None
    roofline = None
    if top:
        kind, amount = work[top]
        ms_step = per_class[top][0]
        if kind == "flop":
            ach, peak, unit, bound = amount / (ms_step * 1e-3) / 1e12, peaks["tensor"], "TFLOP/s", "tensor"
        else:
            ach, peak, unit, bound = amount / (ms_step * 1e-3) / 1e9, peaks["hbm"], "GB/s", "hbm"
        traffic = None
        try:
            ent = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(top)
            if ent and name == "large":
                traffic = ent["bytes_per_launch"]
        except Exception:
            pass
        roofline = {"bound": bound, "kernel_class": top, "achieved": ach, "peak": peak, "unit": unit,
                    "frac": ach / peak, "traffic": traffic, "peak_source": peaks["src"],
                    "ms_per_step_in_class": ms_step, "launch_groups_per_step": per_class[top][1],
                    "class_ms_per_step": {n: round(v[0], 4) for n, v in per_class.items()},
                    "whole_step_tflops": flops_per_token(c) * T * B / (dev_ms / K * 1e-3) / 1e12}
    line = {
        "metric": METRIC, "value": tokens / (dev_ms * 1e-3), "unit": "tokens/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands, f32 accumulate/state" if args.engine == "tc" else "f32", "data": "synthetic",
        "config": bench_config(name, c, world, args.engine, getattr(tr, "transport", None), "B200",
                               "end of step" if args.strict_update else
                               "lazy: layers >= 1 and fc.W updated beside the next step's forward recurrences; every step's "
                               "update (incl. the last, flushed) inside the timed region"),
        "e2e": {"value": tokens / (e2e_wall_ms * 1e-3), "unit": "tokens/s", "ms_per_step": e2e_wall_ms / K,
                "h2d_bytes_per_step": 2 * T * B * 8, "d2h_bytes_per_step": 8,
                "api": "zaremba_b200.Trainer.train_step_host -> zrb_train_step_host"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "final_loss": loss_after,
        "flops_per_token": flops_per_token(c),
        "keep_clipped_grads_mode": {"ms_per_step": keep_ms / K, "value": tokens / (keep_ms * 1e-3),
                                    "note": "same step with coef*g stored back into .grad like clip_grad_norm_ "
                                            "(main.py:115); `value` is the default mode that skips the dead store"},
    }
    if dp_check is not None:
        line["dp_check"] = dp_check
    if not args.no_gpu_baseline:
        # the north_star's bar on the same GPU, timed right after ours with its own clock sample
        s2 = ClockSampler(local)
        s2.start()
        gb = gpu_baseline_leg(c)
        gb["clocks"] = s2.stop()
        line["gpu_baseline"] = gb
        line["vs_baseline"] = line["value"] / gb["value"]
        line["vs_baseline_note"] = ("value / gpu_baseline.value: BASELINE.md publishes no tokens/s; the bar the "
                                    "north_star names is the reference's cuDNN path on the same B200 (single device: "
                                    "the reference has no multi-GPU path), measured in this run")
        line["e2e"]["vs_gpu_baseline"] = line["e2e"]["value"] / gb["value"]
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"], _ = cpu_port_leg(c, args.cpu_budget)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the process's real stdout; everything libraries print while the bench runs (NCCL's
    "NCCL version ..." banner, for one) was diverted to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                       # fd 1 -> stderr for the duration of the run
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--config", default="large", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default=os.environ.get("ZRB_ENGINE", "tc"), choices=["tc", "simt"])
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU work for the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--strict-update", action="store_true",
                    help="apply every weight update at the end of its own step (no lazy update beside the next forward)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the last step's loss, norm, states and (sampled) parameters "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3)
    c = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, c, args.config)
    else:
        run_ours(args, c, args.config)


if __name__ == "__main__":
    main()
