#!/usr/bin/env python
"""
bench.py -- facet->subgrid contributions per second of the B200 SwiFTly hot path.

    python bench.py --gpus N --steps K --warmup W            (this repo, CUDA)
    python bench.py --impl reference --gpus N ...            (reference algorithm on host cores)

One "step" is one COMPLETE forward transform (stages 1-6 of SURVEY.md section 3.2: prepare all
facets, every subgrid column, every subgrid, masks; at N > 1 including the strip exchange)
of the workload, default BASELINE cfg4: N=65536, 8x8 facets of 8192^2 -> 32x32 subgrids of
2048^2, complex128, dense synthetic facets.  metric = (#facets x #subgrids) / step time.

Timing: every step is bracketed by barrier + synchronize and timed with CUDA events on the
compute stream; the step time is the max over ranks; ms_per_step is the mean over the K
timed steps.  Stage 1 consumes the facets (on one GPU the prepared facets reuse their
storage: 64 GiB + 128 GiB do not fit 180 GB otherwise), so facets are regenerated on the
device between steps, outside the timed region.  All inputs are far larger than L2.
Prints ONE JSON line on rank 0.
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (swift config key, description)
    "cfg1": "1k[1]-n512-256",
    "cfg2": "8k[1]-n4k-2k",
    "cfg3": "32k[1]-n8k-4k",
    "cfg4": "64k[1]-n16k-4k",
    # BASELINE "sparse-facet" config: cfg4 geometry, 25 % of the facets (central 4 x 4 block)
    "cfg5": "64k[1]-n16k-4k",
}
SPARSE_BLOCKS = {"cfg5": [0, 8192, 49152, 57344]}
METRIC = "facet->subgrid contributions/sec"
UNIT = "contributions/s"


def note(msg):
    """Progress line on stderr (stdout carries only the JSON line)."""
    if int(os.environ.get("RANK", "0")) == 0:
        sys.stderr.write(f"[bench {time.strftime('%H:%M:%S')}] {msg}\n")
        sys.stderr.flush()


def workload_params(name):
    from ska_sdp_distributed_fourier_transform_b200.swift_configs import SWIFT_CONFIGS

    return dict(SWIFT_CONFIGS[WORKLOADS[name]])


def host_cores():
    """CPU cores this process may actually use: min(affinity, cgroup quota, cpu_count).

    The GPU boxes report 128 CPUs but run in a container limited to 16 CPUs / 200 GiB;
    starting 128 numpy workers there exhausts the memory limit.
    """
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def measured_traffic(kernel_name, world):
    """DRAM bytes per launch of the named kernel from the committed ncu capture (N=1 only)."""
    if world != 1:
        return None
    import glob

    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")), reverse=True):
        try:
            with open(path) as f:
                table = json.load(f)
        except (OSError, ValueError):
            continue
        for key, val in table.items():
            if not key.startswith("_") and key in kernel_name:
                return val["dram_bytes_per_launch"]
    return None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ====================================================================== clocks sampler
class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling during the timed region."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "200", "-i", str(self.gpu_index)],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        power = []
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        clocks, maxc, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    clocks.append(float(parts[1]))
                    maxc.append(float(parts[2]))
                except ValueError:
                    continue
                try:
                    power.append(float(parts[3]))
                except ValueError:
                    pass
                for name, val in zip(names, parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except OSError:
            pass
        if clocks:
            # samples under load: the busy half of the distribution
            out["sm_mhz"] = float(numpy.median(clocks))
            out["sm_max_mhz"] = float(max(maxc))
            out["samples"] = len(clocks)
            out["sm_mhz_min"] = float(min(clocks))
            out["sm_mhz_p10"] = float(numpy.percentile(clocks, 10))
            if power:
                out["power_w_median"] = float(numpy.median(power))
                out["power_w_max"] = float(max(power))
        out["reasons"] = sorted(reasons)
        return out


# ====================================================================== CPU arm
def cpu_baseline_entry(params, cores, steps=1, warmup=0, budget_s=200.0):
    """The reference algorithm RUNNING on the host cores (oracle/cpu_arm.py): one timed
    subgrid column of the forward transform per step -- real shapes, reference task order,
    all cores -- no unit-cost model.

    A step normally covers ``cores`` facets (one facet task per core).  When the caller asks for
    so many steps that this would take longer than ``budget_s`` in total, the first (warm-up)
    step measures the cost per contribution and the timed steps use fewer facets, each split
    into row blocks so that every core still has work; what was run is stated in ``sample``.
    """
    from oracle.cpu_arm import run_column_slice

    N, yB = params["N"], params["yB_size"]
    F = (-(-N // yB)) ** 2
    nf = max(1, min(F, cores))
    chunks = 1
    probe = None
    if warmup > 0 or steps > 1:
        probe = run_column_slice(params, cores, max_facets=nf)
        need = probe["wall_s"] * max(1, steps)
        if need > budget_s:
            nf = max(2, min(nf, int(nf * budget_s / need)))
            chunks = -(-cores // nf)
    runs = [run_column_slice(params, cores, max_facets=nf, chunks=chunks)
            for _ in range(max(1, steps))]
    rate = float(numpy.mean([r["rate"] for r in runs]))
    last = runs[-1]
    entry = {"value": rate, "unit": UNIT, "cores": cores, "kind": last["kind"],
             "sample": last["sample"], "steps": len(runs),
             "step_wall_s": [r["wall_s"] for r in runs],
             "phase_a_s": last["phase_a_s"], "phase_b_s": last["phase_b_s"]}
    if probe is not None:
        entry["full_size_probe"] = {"rate": probe["rate"], "wall_s": probe["wall_s"],
                                    "contributions": probe["contributions"]}
    return entry


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    params = workload_params(args.workload)
    cores = args.cpu_cores or host_cores()
    entry = cpu_baseline_entry(params, cores, steps=max(1, args.steps),
                               warmup=max(0, min(args.warmup, 1)))
    line = {
        "impl": "reference", "metric": METRIC, "value": entry["value"], "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * float(numpy.mean(entry["step_wall_s"])),
        "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64 (complex128)",
        "data": "synthetic", "config": workload_config(args.workload, params, args.gpus),
        "cpu_baseline": entry,
        "e2e": {"value": entry["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_facet_offsets(name):
    """Facet mid-point offsets of a sparse workload (None: full cover)."""
    block = SPARSE_BLOCKS.get(name)
    if block is None:
        return None
    return [(a, b) for a in block for b in block]


def workload_config(name, params, gpus):
    N, yB, xA = params["N"], params["yB_size"], params["xA_size"]
    nf = -(-N // yB)
    ns = -(-N // xA)
    sparse = workload_facet_offsets(name)
    n_facets = nf * nf if sparse is None else len(sparse)
    facets = (f"{nf}x{nf} facets" if sparse is None else
              f"{n_facets} of {nf * nf} facets (central block, offsets {SPARSE_BLOCKS[name]}^2)")
    return {
        "workload": f"{name}: 2D N={N}, {facets} of {yB}^2 -> {ns}x{ns} subgrids of "
                    f"{xA}^2, yN={params['yN_size']}, xM={params['xM_size']}, W={params['W']}, "
                    f"complex128, dense standard-normal facets",
        "contributions_per_step": n_facets * ns * ns,
        "parallelism": "1 GPU" if gpus == 1 else f"facet rows sharded over {gpus} GPUs, "
                       "strips exchanged per subgrid batch",
        "l2": "inputs (>= 64 GiB/step) far larger than the 126 MB L2; no flush needed",
        "timing": "per-step CUDA events, facets regenerated on device between steps (untimed)",
    }


# ====================================================================== GPU arm
def dump_outputs(directory, name, sample, rank, world):
    """``--dump-outputs``: the sampled results of the last timed step as ``<name>.npy``
    (``<name>_rank<r>.npy`` on more than one GPU), float64 (result, pixel, re / im).  The
    pixels are the same seeded sample of every result, and the inputs of every step come from
    fixed seeds, so two builds can be compared output for output.  The forward sample is
    gathered on the device inside the last timed step (one small gather per subgrid)."""
    os.makedirs(directory, exist_ok=True)
    fname = name if world == 1 else f"{name}_rank{rank}"
    arr = sample.array()
    numpy.save(os.path.join(directory, fname + ".npy"), arr)
    note(f"wrote {fname}.npy {arr.shape} to {directory}")


def main_gpu(args):
    # Everything but the final JSON line goes to stderr -- also what libraries print on the C
    # level (NCCL writes its version banner to stdout when the first communicator is created).
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        line = _main_gpu(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    if line is not None:
        print(json.dumps(line))
        sys.stdout.flush()


def _main_gpu_backward(args, dev, rank, world):
    """``--direction backward``: the subgrid -> facet transform (reference api.py:327-463),
    same JSON schema; metric = (#facets x #subgrids) / step time."""
    import torch

    from ska_sdp_distributed_fourier_transform_b200 import bench_support as bs

    params = workload_params(args.workload)
    note(f"setting up backward {args.workload} on {world} GPU(s)")
    runner = bs.BackwardBenchRunner(params, dev, rank, world)
    hbm_gbs, peak_src = measured_peaks()
    for i in range(args.warmup):
        runner.step(timed=False)
        note(f"warm-up step {i + 1}/{args.warmup} done")
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        sampler.start()
    times = []
    for i in range(args.steps):
        if args.dump_outputs and i == args.steps - 1:
            ms, tasks = runner.step(timed=True, keep=True)
            sample = bs.OutputSample(tasks[0].tensor.shape, len(tasks), dev)
            for j, task in enumerate(tasks):
                sample(j, None, task.tensor)
            del tasks
            times.append(ms)
        else:
            times.append(runner.step(timed=True))
        note(f"timed step {i + 1}/{args.steps}: {times[-1]:.1f} ms "
             f"(subgrids {runner.last_parts[0]:.1f} + finish {runner.last_parts[1]:.1f})")
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "facets", sample, rank, world)
    ms = float(numpy.mean(times))
    parity = None if args.no_selfcheck else runner.selfcheck()
    extra = runner.kernel_rooflines(hbm_gbs) if not args.no_roofline else None
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return None
    cfgd = workload_config(args.workload, params, world)
    cfgd["direction"] = "backward (subgrid -> facet): SwiftlyBackward.add_new_subgrid_task for " \
                        "every subgrid of the cover + finish()"
    cfgd["inputs"] = "32 distinct random subgrids fed cyclically (values do not affect timing)"
    line = {
        "metric": "subgrid->facet contributions/sec", "value": runner.contributions_per_step / (ms * 1e-3),
        "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64 (complex128)", "data": "synthetic", "config": cfgd, "step_ms": times,
        "clocks": clocks, "direction": "backward",
        "max_memory_gib": torch.cuda.max_memory_allocated(dev) / 2**30,
    }
    if parity is not None:
        line["parity_max_rel_err"] = parity["parity_max_rel_err"]
        line["parity_check"] = parity
    if extra:
        line["roofline"] = extra["dominant"]
        line["roofline"]["peak_source"] = peak_src
        line["kernel_rooflines"] = extra["kernels"]
    return line


def _main_gpu(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        # NCCL prints its version banner on STDOUT (NCCL_DEBUG=VERSION in this image); stdout
        # must carry the JSON line only
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    if args.direction == "backward":
        return _main_gpu_backward(args, dev, rank, world)
    from ska_sdp_distributed_fourier_transform_b200 import bench_support as bs

    params = workload_params(args.workload)
    note(f"setting up {args.workload} on {world} GPU(s)")
    runner = bs.ForwardBenchRunner(params, dev, rank, world, exchange=args.exchange,
                                   facet_offsets=workload_facet_offsets(args.workload))
    hbm_gbs, peak_src = measured_peaks()

    # ---- device-resident runs (value) ----------------------------------------------
    for i in range(args.warmup):
        runner.step(timed=False)
        note(f"warm-up step {i + 1}/{args.warmup} done")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    times = []
    sample = None
    for i in range(args.steps):
        if args.dump_outputs and i == args.steps - 1:
            owned = [j for j in range(len(runner.sg_cfgs)) if j % world == rank]
            sample = bs.OutputSample((runner.xA, runner.xA), len(owned), dev)
        times.append(runner.step(timed=True, consumer=sample))
        note(f"timed step {i + 1}/{args.steps}: {times[-1]:.1f} ms")
    clocks = sampler.stop() if rank == 0 else None
    if sample is not None:
        dump_outputs(args.dump_outputs, "subgrids", sample, rank, world)
    ms = float(numpy.mean(times))
    contributions = runner.contributions_per_step
    value = contributions / (ms * 1e-3)

    parity = None
    if not args.no_selfcheck:
        parity = runner.selfcheck()  # raises above 1e-9; collective at N > 1
        note(f"self-check: max rel err {parity['parity_max_rel_err']:.2e} "
             f"({parity['subgrids_checked']} subgrids)")
    extra = {}
    if rank == 0 or world > 1:
        extra = runner.kernel_rooflines(hbm_gbs, step_ms=ms) if not args.no_roofline else {}
    note("kernel rooflines done")
    e2e = None
    if not args.no_e2e:
        e2e = runner.e2e(steps=args.e2e_steps, progress=note)
        note(f"e2e done: {e2e['ms_per_step']:.1f} ms/step")
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline_entry(params, args.cpu_cores or host_cores(), steps=1)
        note("cpu baseline done")
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64 (complex128)",
        "data": "synthetic", "config": workload_config(args.workload, params, world),
        "step_ms": times, "gpu_launches": runner.launches_per_step,
        "clocks": clocks,
    }
    if parity is not None:
        line["parity_max_rel_err"] = parity["parity_max_rel_err"]
        line["parity_check"] = parity
    if world > 1:
        line["config"]["exchange"] = runner.exchange_used
    if extra:
        line["roofline"] = extra["dominant"]
        line["roofline"]["peak_source"] = peak_src
        if args.workload == "cfg4":
            line["roofline"]["traffic"] = measured_traffic(line["roofline"]["kernel"], world)
        line["kernel_rooflines"] = extra["kernels"]
        line["bmin_roofline"] = extra["bmin"]
    if e2e is not None:
        line["e2e"] = e2e
    if cpu is not None:
        line["cpu_baseline"] = cpu
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--direction", default="forward", choices=["forward", "backward"],
                    help="forward = facet -> subgrid (the headline metric); backward = subgrid -> facet")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-selfcheck", action="store_true",
                    help="skip the output parity check that follows the timed steps")
    ap.add_argument("--selfcheck", action="store_true", help="(default) kept for symmetry")
    ap.add_argument("--e2e-steps", type=int, default=1)
    ap.add_argument("--cpu-cores", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed, seeded sample of every result of the last timed step "
                         "to DIR/<name>.npy (float64, at most 64 MB)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "copy", "p2p", "nccl"],
                    help="multi-GPU strip exchange: copy engines on peer memory (auto), TMA "
                         "stores into peer memory, or NCCL all_to_all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the GPU implementation")
    if args.impl == "reference":
        main_reference(args)
    else:
        main_gpu(args)


if __name__ == "__main__":
    main()
