"""bench.py -- CTC fwd+bwd frames/s on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C3] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one fused loss+gradient evaluation of one mini-batch of synthetic logits of the named shape:
three kernels (plan -> softmax rows -> lattice, whose last CTA also sums the costs; the backward of the op is
an elementwise scale of the gradient computed here, SURVEY 3.2).  Labels and lengths are device-resident
(b200ctc_loss_and_grad_dev) and four consecutive steps are replayed as one CUDA graph, so the host issues one
graph launch per four steps.

N > 1 (torchrun, one process per GPU) measures two things:
  * the headline line: every rank owns a mini-batch of the same shape (data-parallel training: utterances never
    cross GPUs), the scalar losses are all-reduced over NCCL -- weak scaling, the same workload at every N;
  * "sharded_c5": BASELINE configs[4] (B=512, T=400-1600) PARTITIONED across the ranks with
    shard.balance_shards (strong scaling), with the all-reduced loss checked against the 1-GPU loss of the
    whole batch inside the run (shard_parity).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ctc_fwd_bwd_frames_per_sec"
UNIT = "frames/s"
N_ROTATE = 16          # distinct acts/grads buffer sets cycled through the timed loop (> L2 in total)
GROUP = 8              # steps per CUDA graph (and per all-reduce message at N > 1); 4 per graph measured 3 % slower on C3
MIN_REGION_MS = 50.0   # N > 1: a timed region shorter than this is repeated until it adds up to it
DUMP_GRAD_ELEMS = 1 << 23   # --dump-outputs: a larger gradient is written as this many sampled elements (32 MB)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="C3", choices=["C1", "C2", "C3", "C4", "C5"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip per_config / decoder / sharded_c5 (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


def measured_traffic(workload_key):
    """DRAM bytes per lattice launch from the committed ncu capture (profiles/r02_traffic.json, C3 only)."""
    if workload_key != "C3":
        return None
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                k = json.load(f)["lattice_kernel"]
            return int(k["dram_bytes_read"]) + int(k["dram_bytes_write"])
        except Exception:
            continue
    return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons during the timed region (NVML; nvidia-smi fallback)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.active = threading.Event()          # set while the timed region runs: only those samples count
        self.ready = threading.Event()           # NVML is initialised and has answered once (its start-up is slow)
        self.sm, self.reasons, self.sm_max = [], set(), None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {
                getattr(pynvml, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(pynvml, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(pynvml, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(pynvml, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            self.ready.set()
            while not self.stop_flag.is_set():
                if self.active.is_set():
                    self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                    try:
                        r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for bit, name in names.items():
                            if r & bit:
                                self.reasons.add(name)
                    except Exception:
                        pass
                # every 4 ms: an NVML query holds a driver lock that kernel launches also take (worse with more
                # GPUs in the box) -- at 1 kHz the sampler itself cost one rank of two 7 % of its timed region
                time.sleep(0.004)
        except Exception:
            self.ready.set()
            self._smi()

    def _smi(self):
        import subprocess
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag.is_set():
            if not self.active.is_set():
                time.sleep(0.001)
                continue
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.sm.append(int(f[0])); self.sm_max = int(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                break
            time.sleep(0.1)

    def sample_now(self):
        """One sample taken by the caller's thread (the GPU is busy: the caller keeps its queue full)."""
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
            if self.sm_max is None:
                self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for bit, name in ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
                              (0x4, "sw_power_cap")):
                if r & bit:
                    self.reasons.add(name)
            return True
        except Exception:
            pass
        try:
            import subprocess
            out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
            f = [x.strip() for x in out.strip().split(",")]
            self.sm.append(int(f[0])); self.sm_max = int(f[1])
            return True
        except Exception:
            return False

    def result(self):
        self.stop_flag.set()
        self.join(timeout=5)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def _host_threads():
    """All the host cores this process may use (torchrun exports OMP_NUM_THREADS=1: ignore it)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def config_dict(wl, frames, total_bytes, world):
    """The workload description both arms (--impl b200 / reference) print: identical keys and values."""
    return {"workload": wl.name, "per_gpu_batch": int(wl.B), "frames_per_step_per_gpu": int(frames),
            "algorithmic_bytes_per_step_per_gpu": int(total_bytes), "n_gpus": int(world),
            "parallelism": "utterance-sharded dp%d, scalar loss all-reduce" % world}


def cpu_baseline(wl, acts_np, budget_s=12.0):
    """The oracle's C++/OpenMP restatement of the warp-ctc CPU path (float), timed on this host."""
    from oracle import ctc_cpu
    threads = _host_threads()
    ctc_cpu.ctc_cpu(acts_np[:, :min(8, wl.B)], *_slice(wl, min(8, wl.B)))      # warm-up (page in, build)
    reps, t0 = 0, time.perf_counter()
    while True:
        ctc_cpu.ctc_cpu(acts_np, wl.labels, wl.act_lens, wl.label_lens, precision="f32", num_threads=threads)
        reps += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or reps >= 20:
            break
    frames = int(wl.act_lens.sum())
    return {"value": frames * reps / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d full mini-batches of %s (%d frames each), C++/OpenMP fp32 restatement of the "
                      "warp-ctc CPU path" % (reps, wl.name, frames)}


def torch_cpu_ctc_loss(wl, acts_t, budget_s=8.0):
    """Second CPU data point (BASELINE.md section 4): torch.nn.functional.ctc_loss forward+backward, CPU fp32,
    on the first utterances of the mini-batch (a bounded sample)."""
    import torch
    nb = min(wl.B, 16)
    labels, act_lens, label_lens = _slice(wl, nb)
    x = acts_t[:, :nb].clone().requires_grad_(True)
    tl = torch.from_numpy(labels.astype(np.int64))
    il, ll = torch.from_numpy(act_lens.astype(np.int64)), torch.from_numpy(label_lens.astype(np.int64))
    threads = _host_threads()
    torch.set_num_threads(threads)

    def once():
        lp = torch.log_softmax(x, dim=2)
        loss = torch.nn.functional.ctc_loss(lp, tl, il, ll, blank=0, reduction="sum")
        x.grad = None
        loss.backward()

    once()
    reps, t0 = 0, time.perf_counter()
    while True:
        once()
        reps += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or reps >= 10:
            break
    frames = int(act_lens.sum())
    return {"value": frames * reps / dt, "unit": UNIT, "threads": threads,
            "sample": "%d x forward+backward of the first %d utterances of %s (%d frames), log_softmax + "
                      "torch.nn.functional.ctc_loss, CPU fp32" % (reps, nb, wl.name, frames)}


def _slice(wl, nb):
    L = int(wl.label_lens[:nb].sum())
    return wl.labels[:L], wl.act_lens[:nb], wl.label_lens[:nb]


def dump_outputs(out_dir, costs, loss_sum, grads):
    """--dump-outputs: what a caller of the timed path receives from its last step, as float32 .npy files:
    costs[B], loss_sum[1] and grads[T,B,V].  A gradient of more than DUMP_GRAD_ELEMS elements is written as
    grads_sample.npy, its flat elements at np.sort(np.random.default_rng(0).choice(numel, DUMP_GRAD_ELEMS,
    replace=False)), so that two builds run with the same arguments can be compared output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"costs": costs, "loss_sum": loss_sum}
    grads = torch.as_tensor(grads)
    if grads.numel() <= DUMP_GRAD_ELEMS:
        arrays["grads"] = grads
    else:
        idx = np.sort(np.random.default_rng(0).choice(grads.numel(), DUMP_GRAD_ELEMS, replace=False))
        arrays["grads_sample"] = grads.reshape(-1)[torch.from_numpy(idx).to(grads.device)]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), torch.as_tensor(a).detach().cpu().numpy().astype(np.float32))


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  warp-ctc itself is not in
    /root/reference (un-vendored, un-pinned), so the oracle's C++/OpenMP port is timed, with all the
    host threads, on the same workload, one full mini-batch per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from pytorch_end2end_speech_recognition_b200 import workloads
    from oracle import ctc_cpu
    wl = workloads.make_lengths_and_labels(args.workload)
    acts = workloads.make_acts(wl).numpy()
    frames = int(wl.act_lens.sum())
    threads = _host_threads()
    for _ in range(max(args.warmup, 1)):
        ctc_cpu.ctc_cpu(acts, wl.labels, wl.act_lens, wl.label_lens, precision="f32", num_threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        costs, grads = ctc_cpu.ctc_cpu(acts, wl.labels, wl.act_lens, wl.label_lens, precision="f32", num_threads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, costs, np.array([costs.sum(dtype=np.float64)]), grads)
    value = frames * args.steps / dt
    total, strict, _ = workloads.algorithmic_bytes(wl)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(wl, frames, total, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "one full mini-batch per step (rank 0 only; the CPU path does not shard); C++/OpenMP fp32 "
                                   "restatement of the warp-ctc CPU path (warp-ctc is not vendored in the reference)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


class Runner:
    """The timed object: rotating acts/grads buffer sets (> L2 in total), device-resident labels and lengths,
    GROUP consecutive steps captured as one CUDA graph; at N > 1 the GROUP losses of a graph travel in one
    asynchronous all-reduce (NCCL's own stream) while the next graphs compute."""

    def __init__(self, wl, dev, world, rank, acts_host=None, acts_dev=None, use_graph=True):
        import torch
        import pytorch_end2end_speech_recognition_b200 as b200
        from pytorch_end2end_speech_recognition_b200 import workloads
        self.torch, self.b200, self.wl, self.dev, self.world = torch, b200, wl, dev, world
        acts_bytes = wl.T * wl.B * wl.V * 4
        n_rot = max(2, min(N_ROTATE, int(np.ceil(160e6 / acts_bytes)))) if acts_bytes < 160e6 else 2
        self.group = min(GROUP, n_rot)
        n_rot = (n_rot + self.group - 1) // self.group * self.group
        self.n_rot, self.acts_bytes = n_rot, acts_bytes
        if acts_dev is None:
            self.acts_host = acts_host if acts_host is not None else [
                workloads.make_acts(wl, copy_index=rank * N_ROTATE + i) for i in range(n_rot)]
            self.acts_dev = [a.to(dev) for a in self.acts_host]
        else:
            self.acts_host, self.acts_dev = None, acts_dev
        self.grads_dev = [torch.empty_like(a) for a in self.acts_dev]
        self.costs = torch.empty(wl.B, device=dev)
        Lmax = int(wl.label_lens.max(initial=0))
        ys = np.zeros((wl.B, max(Lmax, 1)), np.int32)
        off = 0
        for b, L in enumerate(wl.label_lens):
            ys[b, :L] = wl.labels[off:off + L]
            off += L
        self.ys = torch.from_numpy(ys).to(dev)
        self.al = torch.from_numpy(wl.act_lens.astype(np.int32)).to(dev)
        self.ll = torch.from_numpy(wl.label_lens.astype(np.int32)).to(dev)
        self.loss_groups = [torch.zeros(self.group, device=dev) for _ in range(2)]
        self.pending = [None, None]
        self.n_groups_done = 0
        self.last_step = None                 # (buffer set, loss group, slot) of the last step run()
        self.graphs = None
        self.launches_per_step = 3            # plan, softmax rows, lattice (+ cost sum in its last CTA)
        # long steps (C4, C5: two buffer sets, 0.7-0.9 ms per step) are issued eagerly: the host needs ~0.02 ms per
        # call, and a graph that holds only two steps costs ~0.04 ms per step at its boundaries (tools/step_probe.py)
        if use_graph and self.group >= 4:
            self._capture()

    def one(self, j, slot):
        self.b200.ctc_loss_and_grad(self.acts_dev[j], self.ys, self.al, self.ll, grads=self.grads_dev[j],
                                    costs=self.costs, loss_sum=slot)

    def _capture(self):
        torch = self.torch
        n_sets = self.n_rot // self.group                       # groups of buffer sets
        n_graphs = n_sets if n_sets % 2 == 0 else 2 * n_sets    # even: graph k writes loss group k % 2
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        graphs = []
        with torch.cuda.stream(side):
            self.one(0, self.loss_groups[0][0:1])               # allocations (workspace of this stream) happen here
            torch.cuda.synchronize()
            for g in range(n_graphs):
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr, stream=side):
                    for k in range(self.group):
                        self.one((g % n_sets) * self.group + k, self.loss_groups[g % 2][k:k + 1])
                graphs.append(gr)
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize()
        self.graphs = graphs

    def _group(self, gi, eager):
        """Steps gi*GROUP .. gi*GROUP+GROUP-1 (one graph replay), then the all-reduce of their losses."""
        import torch.distributed as dist
        g = gi % 2
        if self.world > 1 and self.pending[g] is not None:      # a loss group is rewritten only after its all-reduce
            self.pending[g].wait()
            self.pending[g] = None
        if self.graphs is not None and not eager:
            self.graphs[gi % len(self.graphs)].replay()
        else:
            for k in range(self.group):
                self.one((gi * self.group + k) % self.n_rot, self.loss_groups[g][k:k + 1])
        if self.world > 1:
            self.pending[g] = dist.all_reduce(self.loss_groups[g], async_op=True)   # the one exchange step of the path

    def run(self, steps, eager=False):
        """Exactly `steps` steps."""
        import torch.distributed as dist
        full, rest = divmod(steps, self.group)
        for _ in range(full):
            self._group(self.n_groups_done, eager)
            self.last_step = ((self.n_groups_done * self.group + self.group - 1) % self.n_rot, self.n_groups_done % 2,
                              self.group - 1)
            self.n_groups_done += 1
        if rest:
            g = self.n_groups_done % 2
            if self.world > 1 and self.pending[g] is not None:
                self.pending[g].wait()
                self.pending[g] = None
            for k in range(rest):
                self.one((self.n_groups_done * self.group + k) % self.n_rot, self.loss_groups[g][k:k + 1])
            if self.world > 1:
                self.pending[g] = dist.all_reduce(self.loss_groups[g], async_op=True)
            self.last_step = ((self.n_groups_done * self.group + rest - 1) % self.n_rot, g, rest - 1)
            self.n_groups_done += 1

    def drain(self):
        for g in range(2):
            if self.pending[g] is not None:
                self.pending[g].wait()
                self.pending[g] = None

    def last_loss(self):
        return self.loss_groups[(self.n_groups_done - 1) % 2]


def make_timer(torch, dist, dev, world):
    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, drain):
        """Device time of fn() + drain() between two barriers; max over ranks."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        fn()
        drain()                          # every all-reduce issued in the timed region completes inside it
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms
    return barrier, timed


def measure(runner, timed, steps, warmup, world):
    """W warm-up steps, then K timed steps; at N > 1 a region shorter than MIN_REGION_MS is repeated (same K
    steps each time) and the per-step time is the mean over the repeats."""
    runner.run(warmup)
    runner.drain()
    ms = timed(lambda: runner.run(steps), runner.drain)
    repeats = 1
    if world > 1 and ms < MIN_REGION_MS:
        repeats = int(min(200, np.ceil(MIN_REGION_MS / max(ms, 1e-3))))
        ms = timed(lambda: [runner.run(steps) for _ in range(repeats)], runner.drain) / repeats
    return ms / steps, repeats


def kernel_times(runner, ctc_mod, n_prof):
    """Per-kernel device time: CUDA events inside the C library around each kernel, eager calls."""
    ctc_mod.set_profiling(True)
    k_ms = np.zeros(3)
    slot = runner.loss_groups[0][0:1]
    for i in range(n_prof):
        runner.one(i % runner.n_rot, slot)
        k_ms += np.array(ctc_mod.last_kernel_ms())
    ctc_mod.set_profiling(False)
    return k_ms / n_prof


def roofline_of(wl, workloads, k_ms, ms_per_step, workload_key):
    total_bytes, strict_bytes, frames = workloads.algorithmic_bytes(wl)
    lattice_bytes = total_bytes - int(np.sum(8 * wl.act_lens.astype(np.int64) * wl.V))
    peak, peak_kind = peaks()
    lattice_gbs = lattice_bytes / (k_ms[1] * 1e-3) / 1e9 if k_ms[1] > 0 else 0.0
    return {"bound": "hbm", "kernel": "lattice (alpha/beta recursion + occupancy update)",
            "achieved": lattice_gbs, "peak": peak, "peak_kind": peak_kind + " hbm copy GB/s", "unit": "GB/s",
            "frac": lattice_gbs / peak, "traffic": measured_traffic(workload_key),
            "kernel_ms": {"softmax_rows": k_ms[0], "lattice_and_cost_sum": k_ms[1],
                          "apply_occupancy": (k_ms[2] if wl.V >= 129 else 0.0)},       # large vocabularies only (gathered mode)
            "algorithmic_bytes_per_launch": lattice_bytes,
            "ns_per_frame_of_the_longest_utterance": ms_per_step * 1e6 / max(int(wl.act_lens.max()), 1),
            "whole_step": {"algorithmic_bytes": total_bytes, "strict_dram_bytes": strict_bytes,
                           "achieved": total_bytes / (ms_per_step * 1e-3) / 1e9,
                           "frac": total_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                           "frac_of_8000": total_bytes / (ms_per_step * 1e-3) / 1e9 / 8000.0}}


def per_config_lines(args, torch, dist, dev, timed, ctc_mod, workloads, headline):
    """C1..C5 at N = 1 (20 steps each, same method as the headline): ms/step, roofline fraction, ns/frame and a
    3 s CPU-baseline sample -- so that the driver's record carries all five configs."""
    out = []
    for key in ("C1", "C2", "C3", "C4", "C5"):
        if key == args.workload:
            out.append(headline)
            continue
        wl = workloads.make_lengths_and_labels(key)
        runner = Runner(wl, dev, 1, 0)
        ms, _ = measure(runner, timed, 20, 3, 1)
        k_ms = kernel_times(runner, ctc_mod, 6)
        r = roofline_of(wl, workloads, k_ms, ms, key)
        frames = int(wl.act_lens.sum())
        line = {"workload": wl.name, "key": key, "ms_per_step": ms, "frames_per_sec": frames / (ms * 1e-3),
                "utterances_per_sec": wl.B / (ms * 1e-3), "kernel_ms": r["kernel_ms"], "lattice_frac": r["frac"],
                "whole_step_frac": r["whole_step"]["frac"], "whole_step_frac_of_8000": r["whole_step"]["frac_of_8000"],
                "ns_per_frame_of_the_longest_utterance": r["ns_per_frame_of_the_longest_utterance"]}
        out.append(line)
        del runner
        ctc_mod.release_workspaces()
        torch.cuda.empty_cache()
    return out


def text_like_line(torch, dev, timed, ctc_mod, workloads):
    """The headline shape (C3) with text-like label statistics instead of uniform ones: symbol k drawn with
    p_k ~ 1/k (the most frequent symbol carries a quarter of the labels, as the space does in English
    transcripts).  Informational: the reducers cut the slot range of a frequent symbol into pieces
    (lattice_fast.cuh, reducer groups); without that this workload ran 28 % slower than the uniform one."""
    wl0 = workloads.make_lengths_and_labels("C3")
    rng = np.random.RandomState(5)
    pk = 1.0 / (np.arange(wl0.V - 1) + 1.0)
    pk /= pk.sum()
    wl = wl0._replace(labels=(1 + rng.choice(wl0.V - 1, size=wl0.labels.size, p=pk)).astype(np.int32),
                      name=wl0.name + ", labels ~ 1/k")
    runner = Runner(wl, dev, 1, 0)
    ms, _ = measure(runner, timed, 20, 3, 1)
    del runner
    ctc_mod.release_workspaces()
    torch.cuda.empty_cache()
    return {"workload": wl.name, "ms_per_step": ms, "frames_per_sec": int(wl.act_lens.sum()) / (ms * 1e-3)}


def decoder_line(torch, dev, timed, workloads, b200, key):
    """Greedy decoder (north_star kernel 4): frames/s and fraction of the HBM peak on the logits of `key`
    (bytes = 4*B*T*V read + 4*B*T written)."""
    wl = workloads.make_lengths_and_labels(key)
    n = max(2, int(np.ceil(160e6 / (wl.T * wl.B * wl.V * 4)))) if wl.T * wl.B * wl.V * 4 < 160e6 else 2
    logits = [workloads.make_acts(wl, copy_index=100 + i).transpose(0, 1).contiguous().to(dev) for i in range(n)]
    lens = torch.from_numpy(wl.act_lens.astype(np.int32)).to(dev)
    for i in range(n + 4):                     # every buffer touched once, allocator warm
        b200.greedy_decode(logits[i % n], lens)
    steps = 100
    def calls():                               # results dropped call by call, as a caller would (a list of 100 live
        for i in range(steps):                 # outputs makes every call a cudaMalloc: 5 ms per call, not the decoder)
            b200.greedy_decode(logits[i % n], lens)
    ms = timed(calls, lambda: None) / steps
    frames = int(wl.act_lens.sum())
    nbytes = 4 * frames * wl.V + 4 * frames
    peak, _ = peaks()
    return {"workload": wl.name, "ms_per_call": ms, "frames_per_sec": frames / (ms * 1e-3),
            "algorithmic_bytes": nbytes, "achieved_gbs": nbytes / (ms * 1e-3) / 1e9,
            "frac": nbytes / (ms * 1e-3) / 1e9 / peak, "launches_per_call": 2,
            "note": "through the public call (two output tensors allocated per call); a call costs the host ~0.03 ms, which bounds the small-vocabulary case"}


def sharded_c5(args, torch, dist, dev, world, rank, timed, workloads, b200):
    """BASELINE configs[4]: ONE C5 batch (B=512, T=400-1600) partitioned across the ranks by
    shard.balance_shards (strong scaling; the reference's unused stubs utils/parallel.py:14-33,
    utils/dataset/base.py:260-264).  Every rank evaluates its length-balanced shard; the only exchange is the
    scalar loss.  The all-reduced loss is compared with the loss of the whole batch evaluated on one GPU."""
    from pytorch_end2end_speech_recognition_b200 import shard
    wl = workloads.make_lengths_and_labels("C5")
    index = shard.balance_shards(wl.act_lens, wl.label_lens, wl.V, world)[rank]
    flat, ll, al = shard.shard_batch(wl.labels, wl.label_lens, wl.act_lens, index)
    t_loc = int(al.max())
    swl = workloads.Workload(wl.name + " shard %d/%d" % (rank, world), t_loc, len(index), wl.V, flat, ll, al, wl.seed)
    shard_bytes = t_loc * len(index) * wl.V * 4
    n_rot = max(2, min(N_ROTATE, int(np.ceil(160e6 / shard_bytes))))
    n_rot = (n_rot + GROUP - 1) // GROUP * GROUP
    sel = torch.as_tensor(index, device=dev)
    gen = torch.Generator(device=dev)
    acts_dev, whole0 = [], None
    for i in range(n_rot):
        gen.manual_seed(wl.seed + 7919 * i)                  # the same full batch on every rank, sliced per rank
        full = torch.randn(wl.T, wl.B, wl.V, generator=gen, device=dev)
        if i == 0 and rank == 0:
            whole0 = full
        acts_dev.append(full[:t_loc].index_select(1, sel).contiguous())
        del full
    runner = Runner(swl, dev, world, rank, acts_dev=acts_dev)
    # parity: sum over ranks of the shard losses of buffer set 0 == loss of the whole batch on one GPU
    slot = torch.zeros(1, device=dev)
    runner.one(0, slot)
    total = slot.clone()
    if world > 1:
        dist.all_reduce(total)
    parity = None
    ms_whole = None
    if rank == 0:
        c, loss_whole, _ = b200.ctc_loss_and_grad(whole0, wl.labels, wl.act_lens, wl.label_lens)
        rel = abs(float(total[0]) - float(loss_whole[0])) / abs(float(loss_whole[0]))
        parity = {"allreduced_loss": float(total[0]), "one_gpu_loss": float(loss_whole[0]), "rel_diff": rel, "tol": 1e-5,
                  "ok": bool(rel <= 1e-5)}
        assert parity["ok"], "sharded loss differs from the 1-GPU loss: %r" % (parity,)
        # the whole batch on ONE GPU, timed in the same run (the strong-scaling denominator)
        g = torch.empty_like(whole0)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(2):
            b200.ctc_loss_and_grad(whole0, wl.labels, wl.act_lens, wl.label_lens, grads=g)
        ev0.record()
        for _ in range(5):
            b200.ctc_loss_and_grad(whole0, wl.labels, wl.act_lens, wl.label_lens, grads=g)
        ev1.record()
        torch.cuda.synchronize()
        ms_whole = ev0.elapsed_time(ev1) / 5
        del g, whole0
    ms, repeats = measure(runner, timed, args.steps, args.warmup, world)
    frames = int(wl.act_lens.sum())
    sizes = [len(ix) for ix in shard.balance_shards(wl.act_lens, wl.label_lens, wl.V, world)]
    out = {"workload": wl.name, "scaling": "strong", "n_gpus": world, "ms_per_step": ms, "repeats": repeats,
           "value": frames / (ms * 1e-3), "unit": UNIT, "global_batch": int(wl.B), "utterances_per_rank": sizes,
           "shard_parity": parity, "one_gpu_whole_batch_ms": ms_whole,
           "speedup_vs_one_gpu_whole_batch": (ms_whole / ms) if ms_whole else None,
           "l2": "rotating %d shard buffer sets per rank" % n_rot}
    del runner
    return out


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import pytorch_end2end_speech_recognition_b200 as b200
    from pytorch_end2end_speech_recognition_b200 import ctc as ctc_mod
    from pytorch_end2end_speech_recognition_b200 import workloads

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        warm = torch.zeros(GROUP, device=dev)
        for _ in range(3):
            dist.all_reduce(warm)                 # communicator set-up is not a step
        torch.cuda.synchronize()
    barrier, timed = make_timer(torch, dist, dev, world)

    wl = workloads.make_lengths_and_labels(args.workload)
    frames = int(wl.act_lens.sum())
    total_bytes, strict_bytes, _ = workloads.algorithmic_bytes(wl)
    runner = Runner(wl, dev, world, rank)
    acts_host, acts_bytes, n_rot = runner.acts_host, runner.acts_bytes, runner.n_rot

    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.ready.wait(timeout=5.0)           # NVML start-up (slow, worse with eight ranks) stays out of the timed region
    runner.run(args.warmup)                   # exactly W warm-up steps
    runner.drain()
    sampler.active.set()
    t_host0 = time.perf_counter()
    ms = timed(lambda: runner.run(args.steps), runner.drain)
    host_wall = (time.perf_counter() - t_host0) * 1e3        # wall clock of the same region incl. both barriers (diagnostic)
    repeats = 1
    if world > 1 and ms < MIN_REGION_MS:
        # a multi-rank region of a few milliseconds measures start-up skew, not the step: repeat the K steps
        repeats = int(min(200, np.ceil(MIN_REGION_MS / max(ms, 1e-3))))
        t_host0 = time.perf_counter()
        ms = timed(lambda: [runner.run(args.steps) for _ in range(repeats)], runner.drain) / repeats
        host_wall = (time.perf_counter() - t_host0) * 1e3 / repeats
    host_ms_per_step = host_wall / args.steps
    sampler.active.clear()
    if args.dump_outputs and rank == 0:
        # before any later pass rewrites the shared costs buffer, the loss slots or the gradient buffers
        j, g, k = runner.last_step
        dump_outputs(args.dump_outputs, runner.costs, runner.loss_groups[g][k:k + 1], runner.grads_dev[j])

    def agree_min(n):
        # every rank must take the same branch below: the extra steps contain collectives
        if world == 1:
            return n
        t = torch.tensor([n], device=dev, dtype=torch.int32)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return int(t[0])

    n_in_region = len(sampler.sm)
    if os.environ.get("B200CTC_TEST_CLOCK_SKEW") and rank == 0:
        n_in_region = 0                       # test hook: one rank alone wants the fallback
    n_in_region = agree_min(n_in_region)
    if n_in_region < 3:
        # The timed region lasts ~10 ms and the sampling thread rarely gets the interpreter while the main thread
        # enqueues: take the remaining samples from the main thread under the SAME load right after the timed
        # region (every query is issued with >= 24 steps queued on the GPU).
        for _ in range(12):
            runner.run(24)
            sampler.sample_now()
        runner.drain()
        torch.cuda.synchronize()
    if agree_min(len(sampler.sm)) == 0:
        sampler.active.set()
        timed(lambda: runner.run(max(args.steps, 200)), runner.drain)
        sampler.active.clear()
    clocks = sampler.result()
    clocks["sampled"] = ("in the timed region" if n_in_region >= 3 else
                         "%d in the timed region, the rest under the same load right after it" % n_in_region)
    ms_per_step = ms / args.steps
    value = frames * world / (ms_per_step * 1e-3)

    # host cost of the loop without the barriers: enqueue K steps, do not wait
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    runner.run(args.steps)
    host_enqueue_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    runner.drain()
    torch.cuda.synchronize()

    # ---- per-kernel device time (events inside the C library, separate pass) ----
    k_ms = kernel_times(runner, ctc_mod, min(args.steps, 20))
    roofline = roofline_of(wl, workloads, k_ms, ms_per_step, args.workload)

    # ---- end to end: host buffers, H2D of the step's inputs and D2H of the loss inside the timed region ----
    # Double-buffered input pipeline (what a training loop with a prefetching data loader does): while
    # step i computes, the inputs of step i+1 (logits, padded labels, lengths -- all pinned host memory) travel
    # host -> device.  Every step still pays its own H2D copies and its own D2H read of the loss inside the
    # timed loop.  The logits copy is split in two halves on two copy streams: one stream moves a 12 MB pinned
    # buffer at 17-28 GB/s on this box, two concurrent copies at 53-55 GB/s (PCIe gen5 x16; tools/h2d_bandwidth.py).
    # one pinned allocation for all rotating host buffers: separate pin_memory() calls gave one buffer out of
    # fourteen that copies 2-6x slower than the others on this box (tools/pinned_probe.py)
    pinned_all = torch.empty((len(acts_host),) + tuple(acts_host[0].shape), dtype=acts_host[0].dtype).pin_memory()
    for i, a in enumerate(acts_host):
        pinned_all[i].copy_(a)
    pinned = [pinned_all[i] for i in range(len(acts_host))]
    # labels and lengths of a step: ONE pinned int32 buffer [lengths | label lengths | padded labels] and one copy
    # (three small copies in front of the logits cost that copy stream ~15 us per step)
    B_, Lw = runner.ys.shape
    lab_host = torch.cat([runner.al.cpu(), runner.ll.cpu(), runner.ys.cpu().reshape(-1)]).pin_memory()
    stage = [torch.empty_like(a) for a in runner.acts_dev[:2]]
    lab_dev = [torch.empty_like(lab_host, device=dev) for _ in range(2)]
    stage_lab = [(ld[2 * B_:].view(B_, Lw), ld[:B_], ld[B_:2 * B_]) for ld in lab_dev]
    h2d = acts_bytes + lab_host.numel() * 4
    e2e_loss = []
    n_split = int(os.environ.get("B200CTC_E2E_SPLITS", "2"))
    copy_streams = [torch.cuda.Stream(device=dev) for _ in range(n_split)]
    label_stream = torch.cuda.Stream(device=dev)
    copied = [[torch.cuda.Event() for _ in range(n_split + 1)] for _ in range(2)]
    cuts = [wl.T * k // n_split for k in range(n_split + 1)]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    compute_stream = torch.cuda.current_stream(dev)

    def issue_copy(i):
        d = i % 2
        src = pinned[i % n_rot]
        for k, cs in enumerate(copy_streams):
            with torch.cuda.stream(cs):
                cs.wait_event(consumed[d])                               # the step that last read stage[d] is done
                stage[d][cuts[k]:cuts[k + 1]].copy_(src[cuts[k]:cuts[k + 1]], non_blocking=True)   # H2D of step i's logits, a slice of frames
                copied[d][k].record(cs)
        with torch.cuda.stream(label_stream):
            label_stream.wait_event(consumed[d])
            lab_dev[d].copy_(lab_host, non_blocking=True)                # labels and lengths of step i (device-resident call)
            copied[d][n_split].record(label_stream)

    # The loss of every step is copied device -> host (pinned) right behind its kernels and READ on the host one
    # step later, after the next step has been enqueued: the host never idles the GPU while it prepares a call
    # (what a training loop that logs the previous step's loss does).  Every step's loss is read inside the
    # timed region; the last one after the loop.
    e2e_dev = [torch.empty(1, device=dev) for _ in range(2)]
    e2e_host = [torch.empty(1).pin_memory() for _ in range(2)]
    e2e_read = [torch.cuda.Event(), torch.cuda.Event()]
    # The 4-byte D2H goes on its own stream: on the compute stream it would sit in a copy-engine queue behind
    # the prefetch of the next logits and hold the next step's kernels back by up to one copy (0.1-0.2 ms).
    result_stream = torch.cuda.Stream(device=dev)
    step_done = [torch.cuda.Event(), torch.cuda.Event()]

    def read_loss(i):
        e2e_read[i % 2].synchronize()
        e2e_loss.append(float(e2e_host[i % 2][0]))                      # host read of step i's result

    def e2e_step(i, first):
        d = i % 2
        for ev in copied[d]:
            compute_stream.wait_event(ev)
        b200.ctc_loss_and_grad(stage[d], stage_lab[d][0], stage_lab[d][1], stage_lab[d][2],
                               grads=runner.grads_dev[i % n_rot], costs=runner.costs, loss_sum=e2e_dev[d])
        consumed[d].record(compute_stream)
        if world > 1:
            dist.all_reduce(e2e_dev[d])
        step_done[d].record(compute_stream)
        with torch.cuda.stream(result_stream):
            result_stream.wait_event(step_done[d])
            e2e_host[d].copy_(e2e_dev[d], non_blocking=True)             # D2H of the step's result
            e2e_read[d].record(result_stream)
        issue_copy(i + 1)                                               # next step's inputs travel while this one computes
        if i > first:
            read_loss(i - 1)

    def e2e_run(steps, first):
        # `first`..`first+steps-1`; the copy of step `first` is issued here, inside the timed region
        issue_copy(first)
        for i in range(first, first + steps):
            e2e_step(i, first)
        read_loss(first + steps - 1)
        for cs in copy_streams:
            cs.synchronize()

    for d in (0, 1):
        consumed[d].record(compute_stream)
    e2e_run(n_rot + 2, 0)                     # warm-up: every rotating host buffer has been copied once
    torch.cuda.synchronize()
    e2e_ms = timed(lambda: e2e_run(args.steps, n_rot + 2), lambda: None) / args.steps
    e2e = {"value": frames * world / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms,
           "pipeline": "double-buffered: H2D of step i+1's logits (%d slices on %d copy streams), padded labels and lengths (one copy, own stream) overlaps the kernels of step i; the loss of step i is copied D2H behind its kernels (own stream) and read on the host after step i+1 is enqueued (one extra prefetch copy per run is also inside the timed region)" % (n_split, n_split)}
    del pinned_all, pinned, stage

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(wl, frames, total_bytes, world),
        "details": {"utterances_per_sec": wl.B * world / (ms_per_step * 1e-3), "timed_region_repeats": repeats,
                    "l2": "rotating %d acts/grads buffer sets (%.0f MB > L2)" % (n_rot, 2 * n_rot * acts_bytes / 1e6),
                    "launch": ("device-resident labels/lengths, %d steps per CUDA graph" % runner.group if runner.graphs is not None else
                               "device-resident labels/lengths, eager calls") + "; N > 1: the %d losses of a group of steps in one asynchronous all-reduce" % runner.group},
        "host": {"wall_ms_per_step": host_ms_per_step, "enqueue_ms_per_step": host_enqueue_ms, "cpus": _host_threads()},
        "roofline": roofline, "e2e": e2e, "gpu_launches": runner.launches_per_step * args.steps * repeats, "clocks": clocks,
    }
    headline = {"workload": wl.name, "key": args.workload, "ms_per_step": ms_per_step, "frames_per_sec": value / world,
                "utterances_per_sec": wl.B / (ms_per_step * 1e-3), "kernel_ms": roofline["kernel_ms"],
                "lattice_frac": roofline["frac"], "whole_step_frac": roofline["whole_step"]["frac"],
                "whole_step_frac_of_8000": roofline["whole_step"]["frac_of_8000"],
                "ns_per_frame_of_the_longest_utterance": roofline["ns_per_frame_of_the_longest_utterance"]}
    acts0 = acts_host[0]
    del runner
    ctc_mod.release_workspaces()
    torch.cuda.empty_cache()
    # every GPU measurement first, the CPU legs last: seconds of CPU work leave the GPU idle and its clocks low
    if world == 1 and not args.no_extras:
        out["per_config"] = per_config_lines(args, torch, dist, dev, timed, ctc_mod, workloads, headline)
        out["text_like_labels"] = text_like_line(torch, dev, timed, ctc_mod, workloads)
        out["greedy_decoder"] = [decoder_line(torch, dev, timed, workloads, b200, k) for k in ("C3", "C4")]
    if not args.no_extras:
        out["sharded_c5"] = sharded_c5(args, torch, dist, dev, world, rank, timed, workloads, b200)
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(wl, acts0.numpy())
        out["cpu_torch_ctc_loss"] = torch_cpu_ctc_loss(wl, acts0)
        for line in out.get("per_config", []):
            if line["key"] == args.workload:
                line["cpu_baseline_frames_per_sec"] = out["cpu_baseline"]["value"]
            else:
                w2 = workloads.make_lengths_and_labels(line["key"])
                cb = cpu_baseline(w2, workloads.make_acts(w2).numpy(), budget_s=3.0)
                line["cpu_baseline_frames_per_sec"] = cb["value"]
                line["cpu_baseline_sample"] = cb["sample"]
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True        # running the benchmark adds no __pycache__ to the source tree
    main()
