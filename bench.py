#!/usr/bin/env python3
"""bench.py -- FNO rollout steps/sec on 64x64 cavity fields (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--act bf16|f32]
                    [--dump-outputs DIR]

One "step" = one `generate()` of the whole per-GPU batch (one autoregressive rollout step,
SURVEY.md 8d).  N=1 workload = BASELINE.json configs[1]: cavity (p=5), batch 256, hidden activations
stored as bf16, fp32 arithmetic; the fp32-storage (parity) mode is measured in the same run and reported
under "fp32_storage".  N>1 (torchrun, one rank per GPU): each rank rolls out its own 256 cases, no
data-path collective ("weak" scaling); value = N*K / max-over-ranks time.

The printed JSON line carries, besides the contract keys: "e2e" (public API, HOST buffers, H2D+D2H inside
the timed region every step), "roofline" (dominant kernel, algorithmic bytes / CUDA-event duration /
measured HBM peak), "kernels" (per-kernel mean durations from a second, event-bracketed pass),
"cpu_baseline" (oracle torch port = the reference's own library calls, timed on this host's cores),
"rel_l2" (per-step relative L2 vs the fp32 CPU oracle on identical inputs) and "clocks".

--dump-outputs DIR writes what the timed rollout returned for its last step, for both storage modes, as
DIR/preds_last_step_{bf16,f32}.npy (float32, B x 2 x 64 x 64; rank 0's shard).  Weights and inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

# keep stdout to the single JSON line: NCCL prints its version banner / debug lines to stdout otherwise
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from cfdbench_b200 import dp, synth  # noqa: E402

# roofline.traffic = dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, read at run
# time from the committed summary of the `ncu --set full` capture (profiles/ncu_traffic.json, written by
# tools/summarize_profiles.py from the .ncu-rep).  Keyed by kernel name, activation storage and batch: if the kernel was
# renamed / the workload changed since the capture, the lookup fails and traffic is reported as null with the reason.
def ncu_traffic(kernel: str, act: str, batch: int):
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            table = json.load(f)
    except Exception as e:  # noqa: BLE001
        return None, f"profiles/ncu_traffic.json unreadable ({type(e).__name__})"
    ent = table.get(f"{kernel}|{act}|{batch}")
    if ent is None:
        return None, f"no ncu capture of {kernel} at act={act}, B={batch} in profiles/ncu_traffic.json"
    return int(ent["dram_bytes"]), ent.get("source", "")

METRIC = "fno_rollout_steps_per_sec"
UNIT = "steps/s"
HW = 64 * 64


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def build_model(act: str, p: int, seed: int = 0):
    from cfdbench_b200 import Fno2d, loss_name_to_fn
    sd = synth.make_state_dict(seed, n_params=p)
    m = Fno2d(in_chan=2, out_chan=2, n_case_params=p, loss_fn=loss_name_to_fn("nmse"), num_layers=synth.DEPTH,
              hidden_dim=synth.HIDDEN, modes1=synth.MODES, modes2=synth.MODES,
              act_dtype="bfloat16" if act == "bf16" else "float32")
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    return m, sd


def timed_rollout(model, inp, cp, mk, steps: int, warmup: int, reps: int = 5):
    """K steps = one native rollout of K steps on torch's current stream, CUDA events around it."""
    dev = model.device
    t_spin = time.perf_counter()  # bring the SM clocks up from idle before the contract's W warm-up steps
    while time.perf_counter() - t_spin < 0.4:  # same `steps` as the timed call: its output buffer gets cached
        model.generate_many(inp, cp, mk, steps)
        torch.cuda.synchronize(dev)
    # W warm-up steps, issued as whole rollouts of `steps` steps (>= W steps in total): the timed call then reuses
    # the same captured graph and output buffer, so no capture / allocation lands inside the timed region
    for _ in range(-(-max(warmup, 0) // steps)):
        model.generate_many(inp, cp, mk, steps)
    torch.cuda.synchronize(dev)
    if torch.distributed.is_initialized():
        torch.distributed.barrier()
    torch.cuda.synchronize(dev)
    times = []
    for _ in range(reps):   # every repetition times exactly K steps, barrier + synchronize on both sides
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        seq = model.generate_many(inp, cp, mk, steps)
        e1.record()
        torch.cuda.synchronize(dev)
        if torch.distributed.is_initialized():
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)
        times.append(e0.elapsed_time(e1) / 1e3)
    return times, seq


def timed_e2e(model, batch: dict, steps: int, warmup: int):
    """Public API with HOST buffers: every step copies that step's input frame (+mask, params) H2D from pinned
    memory, runs generate(), and reads the predicted frame back D2H (fno_rollout_host with steps=1)."""
    pin = {k: torch.from_numpy(batch[k]).pin_memory() for k in ("inputs", "case_params", "mask")}
    cur = pin["inputs"]
    for _ in range(max(warmup, 1)):
        model.generate_many(cur, pin["case_params"], pin["mask"], 1)
    torch.cuda.synchronize(model.device)
    t0 = time.perf_counter()
    cur = pin["inputs"]
    for _ in range(steps):
        cur = model.generate_many(cur, pin["case_params"], pin["mask"], 1)[0]  # syncs: result is on the host
    t = time.perf_counter() - t0
    b = batch["inputs"].shape[0]
    h2d = b * (2 + 1) * HW * 4 + batch["case_params"].nbytes
    d2h = b * 2 * HW * 4
    return t, h2d, d2h


def kernel_pass(model, inp, cp, mk, steps: int):
    """Second pass with CUDA events around every kernel launch (same stream, same C-ABI calls as fno_forward issues
    for this model): mean duration per kernel."""
    from cfdbench_b200 import _lib
    lib = _lib.load()
    b = inp.shape[0]
    pk = model._pack()
    ws, bufs = model._workspace(b)
    w = pk["struct"]
    act = model._act_code()
    st = model._stream()
    acts = [bufs["act0"], bufs["act1"]]
    preds = torch.empty(b, 2, 64, 64, device=model.device)
    fused = "ym_img" in bufs
    names = ["lift", "dft_fwd", "mode_mix"] + (["block_fused"] if fused else ["inv_kx", "block_out"]) + ["project"]
    evs = {n: [] for n in names}

    def timed(name, fn):
        a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(fn(), name)
        z.record()
        evs[name].append((a, z))

    cur_in = inp
    inv = 1.0 / HW
    for _ in range(steps):
        timed("lift", lambda: lib.fno_lift_fwd(cur_in.data_ptr(), mk.data_ptr(), cp.data_ptr(), C.byref(w),
                                               acts[0].data_ptr(), b, act, st))
        cur = 0
        for l in range(model.num_layers):
            timed("dft_fwd", lambda: lib.fno_spectral_dft_fwd(acts[cur].data_ptr(), bufs["xm"].data_ptr(), b, act, 1.0, 1.0, st))
            if fused:
                timed("mode_mix", lambda: lib.fno_mode_mix_image(bufs["xm"].data_ptr(), w.spec_wk[l], bufs["ym_img"].data_ptr(), b, st))
                timed("block_fused", lambda: lib.fno_block_fused(bufs["ym_img"].data_ptr(), acts[cur].data_ptr(), w.w0t[l],
                                                                 w.w0_b[l], acts[cur ^ 1].data_ptr(), b, st))
            else:
                timed("mode_mix", lambda: lib.fno_mode_mix(bufs["xm"].data_ptr(), w.spec_wk[l], bufs["ym"].data_ptr(), b, st))
                timed("inv_kx", lambda: lib.fno_spectral_inv_kx(bufs["ym"].data_ptr(), bufs["z"].data_ptr(), b, inv, 2 * inv, st))
                timed("block_out", lambda: lib.fno_block_out(_lib.EPI_GELU, bufs["z"].data_ptr(), acts[cur].data_ptr(),
                                                             w.w0t[l], w.w0_b[l], acts[cur ^ 1].data_ptr(), None, None, b,
                                                             act, st))
            cur ^= 1
        timed("project", lambda: lib.fno_project_fwd(acts[cur].data_ptr(), mk.data_ptr(), C.byref(w), preds.data_ptr(), b, act, st))
        cur_in = preds
    torch.cuda.synchronize(model.device)
    out = {}
    for n in names:
        ms = [a.elapsed_time(z) for a, z in evs[n]]
        out[n] = {"mean_us": 1e3 * float(np.mean(ms)), "launches_per_step": len(ms) // steps}
    return out


def rel_l2_vs_oracle(model, sd, batch, steps: int = 4, nsamp: int = 2):
    """Per-step relative L2 vs the fp32 CPU oracle (torch port == reference library calls) on identical
    inputs (teacher-forced: both get the oracle's previous frame)."""
    from oracle import fno_numpy as onp
    from oracle import fno_torch_port as opt
    pp = opt.params_from_numpy(sd)
    inp = torch.from_numpy(batch["inputs"][:nsamp])
    cp = torch.from_numpy(batch["case_params"][:nsamp])
    mk = torch.from_numpy(batch["mask"][:nsamp])
    out, cur = [], inp
    with torch.no_grad():
        for _ in range(steps):
            ref = opt.forward(pp, cur, cp, mk)["preds"]
            got = model.generate(cur.cuda(), cp.cuda(), mk.cuda()).cpu()
            out.append(onp.rel_l2(got.numpy(), ref.numpy().astype(np.float64)))
            cur = ref
    return out


def timed_train_step(p: int, batch_size: int, steps: int = 5, warmup: int = 3, fused_adam: bool = True,
                     problem: str = "cavity", act: str = "f32"):
    """fwd -> loss["nmse"].backward() -> Adam.step -> zero_grad (reference src/train_auto.py:233-260) on this GPU,
    fp32 storage, data parallel gradient all-reduce when launched under torchrun.  Secondary number, not the metric.
    fused_adam=False uses the optimizer the reference script builds itself (torch.optim.Adam)."""
    from cfdbench_b200 import FusedAdam
    model, _ = build_model(act, p)
    if torch.distributed.is_initialized():
        model.enable_data_parallel()
    batch = synth.make_batch(7, batch_size, problem)
    tb = {k: torch.from_numpy(v).to(model.device) for k, v in batch.items()}
    opt = (FusedAdam if fused_adam else torch.optim.Adam)(model.parameters(), lr=1e-4)
    ev = []
    for i in range(warmup + steps):
        a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = model(**tb)
        out["loss"]["nmse"].backward()
        opt.step()
        opt.zero_grad()
        z.record()
        if i >= warmup:
            ev.append((a, z))
    torch.cuda.synchronize(model.device)
    ms = float(np.median([a.elapsed_time(z) for a, z in ev]))
    dp_mode = getattr(model, "dp_segments", "one")
    del model
    torch.cuda.empty_cache()
    world = torch.distributed.get_world_size() if torch.distributed.is_initialized() else 1
    return _train_result(ms, batch_size, world, problem, fused_adam, act, dp_mode)


def _train_result(ms, batch_size, world, problem, fused_adam, act, dp_mode):
    dp_text = {"one": "ONE NCCL AVG all-reduce of the flat gradient buffer after backward",
               "two": "NCCL AVG in two segments, the first overlapped with the rest of backward",
               "all": "NCCL AVG per gradient segment, overlapped with the rest of backward"}.get(dp_mode, dp_mode)
    return {"value": 1e3 / ms, "unit": "train steps/s per GPU", "ms_per_step": ms, "batch_per_gpu": batch_size,
            "global_batch": batch_size * world, "problem": problem,
            "what": "fwd + native MseLoss + nmse.backward" + (f" + gradient all-reduce ({dp_text})" if world > 1 else "") +
                    " + " + ("FusedAdam (fno_adam_step)" if fused_adam else "torch.optim.Adam") + f".step, {act} storage"}


def host_cpu():
    """(model string, physical cores, logical cpus) of this host."""
    model = "unknown"
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    model = ln.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or os.cpu_count()
    except Exception:  # noqa: BLE001
        phys = os.cpu_count()
    return model, int(phys or 1), int(os.cpu_count() or 1)


def reference_impl(sd):
    """The CPU implementation `cpu_baseline` / `--impl reference` time, as (kind, forward, train_step_factory).
    kind "reference": the UNMODIFIED reference module, byte-compiled by __graft_entry__.build() into the git-ignored
    oracle/_ref/src (oracle/build_ref.py); kind "port": oracle/fno_torch_port.py, verified bit-identical to it by
    oracle/make_golden.py, when oracle/_ref is absent."""
    ref_src = os.path.join(ROOT, "oracle", "_ref", "src")
    if os.path.isdir(os.path.join(ref_src, "models", "fno")):
        try:
            sys.path.insert(0, ref_src)
            rs = torch.random.get_rng_state()
            from models.fno.fno2d import Fno2d as RefFno2d   # seeds the global RNGs at import (fno2d.py:13-14)
            from models.loss import loss_name_to_fn as ref_loss
            torch.random.set_rng_state(rs)
            p = sd["fc0.weight"].shape[1] - 5
            m = RefFno2d(in_chan=2, out_chan=2, n_case_params=p, loss_fn=ref_loss("nmse"), num_layers=synth.DEPTH,
                         hidden_dim=synth.HIDDEN, modes1=synth.MODES, modes2=synth.MODES)
            m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
            m.eval()

            def fwd(inp, cp, mk):
                return m.generate(inputs=inp, case_params=cp, mask=mk)

            def many(inp, cp, mk, steps):
                return m.generate_many(inp, cp, mk, steps)

            def make_train():
                opt_ = torch.optim.Adam(m.parameters(), lr=1e-4)

                def step(tb):
                    out = m(**tb)
                    out["loss"]["nmse"].backward()
                    opt_.step()
                    opt_.zero_grad()
                    return out["loss"]["nmse"].item()
                return step
            return "reference", fwd, many, make_train
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"bench.py: oracle/_ref unusable ({type(e).__name__}: {e}); timing the oracle port\n")
        finally:
            if sys.path and sys.path[0] == ref_src:
                sys.path.pop(0)
    from oracle import fno_torch_port as opt
    pp = opt.params_from_numpy(sd)

    def fwd(inp, cp, mk):
        return opt.forward(pp, inp, cp, mk)["preds"]

    def many(inp, cp, mk, steps):
        return opt.rollout(pp, inp, cp, mk, steps)

    def make_train():
        pg = opt.params_from_numpy(sd, requires_grad=True)
        opt_ = torch.optim.Adam(list(pg.values()), lr=1e-4)
        return lambda tb: opt.train_step(pg, opt_, tb)
    return "port", fwd, many, make_train


def _median_time(fn, n_warm, n_iter, budget_s):
    for _ in range(n_warm):
        fn()
    ts, t_start = [], time.perf_counter()
    while len(ts) < n_iter and (time.perf_counter() - t_start) < budget_s:
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), len(ts)


def cpu_baseline(sd, batch, budget_s: float = 12.0, max_steps: int = 6):
    """The reference's CPU path on this host's cores (SURVEY.md 8d / BASELINE.md section 3): the headline workload
    (B=256 rollout step) on a bounded sample, plus config (1) B=1 single step, the B=1 20-step generate_many of
    test_multistep.py:144-149, the B=8 train step of train_auto.py:233-260, and the 1-thread figure."""
    kind, fwd, many, make_train = reference_impl(sd)
    cpu_model, phys, logical = host_cpu()
    prev_threads = torch.get_num_threads()
    torch.set_num_threads(phys)
    inp, cp, mk = (torch.from_numpy(batch[k]) for k in ("inputs", "case_params", "mask"))
    out = {}
    with torch.no_grad():
        cur = [inp]

        def step256():
            cur[0] = fwd(cur[0], cp, mk)
        med, n = _median_time(step256, 1, max_steps, budget_s)
        out.update({"value": 1.0 / med, "unit": UNIT, "cores": phys, "kind": kind, "cpu_model": cpu_model,
                    "logical_cpus": logical,
                    "sample": f"{n} rollout steps of the same B={inp.shape[0]} cavity batch, fp32, torch {torch.__version__} "
                              f"CPU, {phys} threads, median {med * 1e3:.1f} ms/step"})
        i1, c1, m1 = inp[:1], cp[:1], mk[:1]
        med1, n1 = _median_time(lambda: fwd(i1, c1, m1), 5, 30, 3.0)
        med20, n20 = _median_time(lambda: many(i1[0], c1[0], m1[0, 0] if m1.dim() == 4 else m1[0], 20), 1, 5, 4.0)
        torch.set_num_threads(1)
        med1t, n1t = _median_time(lambda: fwd(i1, c1, m1), 3, 20, 3.0)
        torch.set_num_threads(phys)
    b8 = synth.make_batch(11, 8, "cavity")
    tb8 = {k: torch.from_numpy(v) for k, v in b8.items()}
    train = make_train()
    medt, nt = _median_time(lambda: train(tb8), 2, 10, 4.0)
    out["others"] = {
        "b1_generate_ms": {"median": med1 * 1e3, "iters": n1, "threads": phys},                    # BASELINE config (1)
        "b1_generate_1thread_ms": {"median": med1t * 1e3, "iters": n1t, "threads": 1},
        "b1_generate_many_20_steps_ms": {"median": med20 * 1e3, "iters": n20, "threads": phys},
        "b8_train_step_ms": {"median": medt * 1e3, "iters": nt, "threads": phys,
                             "what": "fwd + nmse.backward + Adam.step + zero_grad + .item()"},
    }
    torch.set_num_threads(prev_threads)
    return out


def dump_outputs(out_dir: str, arrays: dict, limit: int = 64 << 20) -> None:
    """Write every (B, ...) array as out_dir/<name>.npy in float32.  When they would exceed `limit` bytes together, each
    keeps the batch rows np.random.default_rng(0) picks (sorted), the same rows in every run with the same --batch."""
    os.makedirs(out_dir, exist_ok=True)
    budget = limit // max(len(arrays), 1)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        rows = max(budget // (a[0].nbytes or 1), 1)
        if rows < a.shape[0]:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_name(batch: int) -> str:
    return (f"FNO autoregressive rollout, cavity_prop_bc_geo shape (p=5), batch {batch}/GPU, 64x64x2 "
            f"fields, 4 Fourier layers x 32 ch x 12x12 modes (BASELINE.json configs[1])")


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's own CPU implementation of the path (the unmodified module from oracle/_ref when
    build() could compile it, else the verified port) on ALL physical cores of this host -- also under torchrun, where
    OMP_NUM_THREADS=1 would otherwise leave it single-threaded.  Rank 0 only; the other ranks exit."""
    if rank != 0:
        return
    cpu_model, phys, logical = host_cpu()
    torch.set_num_threads(phys)
    p = synth.n_case_params("cavity")
    sd = synth.make_state_dict(0, n_params=p)
    batch = synth.make_batch(1, args.batch, "cavity", with_label=False)
    kind, fwd, _, _ = reference_impl(sd)
    inp, cp, mk = (torch.from_numpy(batch[k]) for k in ("inputs", "case_params", "mask"))
    cur = inp
    with torch.no_grad():
        for _ in range(args.warmup):
            cur = fwd(cur, cp, mk)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cur = fwd(cur, cp, mk)
        t = time.perf_counter() - t0
    val = args.steps / t
    threads = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # same workload as the GPU arm; one step = one pass over one batch of `batch_per_gpu` cases
        "config": {"workload": workload_name(args.batch), "batch_per_gpu": args.batch, "global_batch": args.batch,
                   "act_storage": "f32", "arithmetic": "fp32",
                   "implementation": (f"reference CPU path ({'unmodified src/models/fno/fno2d.py from oracle/_ref' if kind == 'reference' else 'torch port of src/models/fno/fno2d.py'}), "
                                      f"{threads} threads on {cpu_model} ({phys} cores), rank 0 only")},
        "sample_steps_per_s": val * args.batch,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind, "cpu_model": cpu_model,
                         "sample": f"{args.steps} rollout steps, B={args.batch}, torch {torch.__version__} CPU"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="cases per GPU")
    ap.add_argument("--act", default="bf16", choices=["bf16", "f32"], help="headline activation storage")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch every kernel on the stream instead of replaying the rollout from a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the predictions of the last timed rollout step of each storage mode as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    rank, local, world = dp.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    p = synth.n_case_params("cavity")
    batch = synth.make_batch(1 + rank, args.batch, "cavity", with_label=False)  # seed 0(+rank) shards (SURVEY 8d)
    inp, cp, mk = (torch.from_numpy(batch[k]).to(dev) for k in ("inputs", "case_params", "mask"))

    results, last_preds = {}, {}
    sampler = ClockSampler(local)
    for act in ([args.act] + [a for a in ("bf16", "f32") if a != args.act]):
        model, sd = build_model(act, p)
        model.graph_rollout = not args.no_graph
        headline = act == args.act
        if headline and rank == 0:
            sampler.start()
        ts, seq = timed_rollout(model, inp, cp, mk, args.steps, args.warmup, reps=5 if headline else 3)
        if headline and rank == 0:
            clocks = sampler.stop()
        if args.dump_outputs and rank == 0:
            last_preds[act] = seq[-1].cpu()   # a copy: seq[-1] is a view of the whole K-step rollout tensor
        del seq
        ts_max = [dp.max_over_ranks(t, dev) for t in ts]   # max over ranks of every repetition
        r = {"t": float(np.median(ts_max)), "t_min": float(min(ts_max)), "t_all": ts_max}
        if headline:
            # Before any CPU-side oracle work: the intra-op worker threads of a torch CPU op keep spinning for ~200 ms
            # after it returns, and a host loop of ~40 driver calls per step started in that window ran 3-4x slower
            # (238-383 instead of ~1000 steps/s in 3 of 27 runs).  Median of three K-step repetitions.
            reps = [timed_e2e(model, batch, args.steps, 3) for _ in range(3)]
            te, h2d, d2h = sorted(reps)[1]
            r["e2e"] = (dp.max_over_ranks(te, dev), h2d, d2h)
        if rank == 0:
            r["kernels"] = kernel_pass(model, inp, cp, mk, min(args.steps, 5))
            r["rel_l2"] = rel_l2_vs_oracle(model, sd, batch)
        results[act] = r
        del model
        torch.cuda.empty_cache()

    train = timed_train_step(p, min(args.batch, 64))  # all ranks take part (gradient all-reduce under torchrun)
    train["torch_adam_ms_per_step"] = timed_train_step(p, min(args.batch, 64), fused_adam=False)["ms_per_step"]
    # BASELINE.json configs[2]: cylinder (p = 8), 256 cases per GPU (global 2048 on 8 GPUs), data parallel
    train_cyl = timed_train_step(synth.n_case_params("cylinder"), args.batch, problem="cylinder")
    if rank != 0:
        if torch.distributed.is_initialized():
            torch.distributed.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {f"preds_last_step_{a}": t for a, t in last_preds.items()})

    peak, peak_src = measured_hbm_peak()

    def summarize(act):
        r = results[act]
        k = r["kernels"]
        elt = 2 if act == "bf16" else 4
        fused = "block_fused" in k
        dom = "block_fused" if fused else "block_out"
        dom_kernel = "block_fused_kernel" if fused else "block_tc_kernel"
        k3 = k[dom]["mean_us"] * 1e-6
        alg = args.batch * 32 * HW * 2 * elt  # SURVEY 8d: 32*64*64*(s_in+s_out) per sample-layer x samples/launch
        layer = [n for n in ("dft_fwd", "mode_mix", "inv_kx", "block_out", "block_fused") if n in k]
        blk = sum(k[n]["mean_us"] for n in layer) * 1e-6
        step_us = sum(v["mean_us"] * v["launches_per_step"] for v in k.values())
        # SURVEY 8d whole-step algorithmic bytes per sample (layer-fused design): 2,662,400 B with bf16 storage
        step_alg = args.batch * (3 * HW * 2 + 32 * HW * elt + 4 * 32 * HW * 2 * elt + 32 * HW * elt + 2 * HW * 4) if act == "f32" \
            else args.batch * 2662400
        ms = 1e3 * r["t"] / args.steps
        traffic, traffic_src = ncu_traffic(dom_kernel, act, args.batch)
        return {
            "value": world * args.steps / r["t"], "ms_per_step": ms, "ms_per_step_min": 1e3 * r["t_min"] / args.steps,
            "reps_ms_per_step": [1e3 * t / args.steps for t in r["t_all"]],
            "roofline": {"bound": "hbm", "kernel": dom_kernel, "achieved": alg / k3 / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": alg / k3 / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                         "share_of_step": k[dom]["mean_us"] * k[dom]["launches_per_step"] / step_us,
                         "fourier_layer_frac": alg / blk / 1e9 / peak, "fourier_layer_us": blk * 1e6,
                         "step_frac": step_alg / (ms * 1e-3) / 1e9 / peak, "step_algorithmic_bytes": step_alg},
            "kernels": k, "rel_l2": r["rel_l2"],
            "launches_per_step": sum(v["launches_per_step"] for v in k.values()),
        }

    head = summarize(args.act)
    other_act = "f32" if args.act == "bf16" else "bf16"
    other = summarize(other_act)
    te, h2d, d2h = results[args.act]["e2e"]
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if args.act == "bf16" else "f32", "data": "synthetic",
        "config": {
            "workload": workload_name(args.batch),
            "batch_per_gpu": args.batch, "global_batch": args.batch * world,
            "act_storage": "bf16" if args.act == "bf16" else "f32",
            "arithmetic": "fp32-grade: tensor-core products as 3xTF32 / bf16x3 (24-bit operands), fp32 accumulation",
            "parallelism": f"dp{world} (independent case shards, no data-path collective)",
            "l2": "inputs larger than L2: per-step working set (2 activation buffers + modes) = "
                  f"{(2 * args.batch * 32 * HW * (2 if args.act == 'bf16' else 4) + 2 * args.batch * 288 * 32 * 8) / 1e6:.0f} MB > 126 MB",
            "cuda_graph": not args.no_graph,
            "timing": "median of 5 repetitions of K steps each (CUDA events, max over ranks per repetition); "
                      "ms_per_step_min / reps_ms_per_step alongside",
        },
        "sample_steps_per_s": head["value"] * args.batch,
        "ms_per_step_min": head["ms_per_step_min"], "reps_ms_per_step": head["reps_ms_per_step"],
        "e2e": {"value": world * args.steps / te, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": args.steps * head["launches_per_step"],
        "roofline": head["roofline"], "kernels": head["kernels"], "rel_l2": head["rel_l2"],
        ("fp32_storage" if other_act == "f32" else "bf16_storage"): other,
        "train_step": train, "train_step_cylinder": train_cyl,
        "clocks": clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(synth.make_state_dict(0, n_params=p), batch)
    print(json.dumps(line))
    if torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
