"""
Benchmark driver for the forward transform (used by ``bench.py``).

Keeps the measurement logic next to the API it measures: the timed region calls the
public ``SwiftlyForward`` (one GPU) or ``SwiftlyForwardSharded`` (one rank per GPU)
classes, nothing else.
"""

import time

import numpy
import torch
import torch.distributed as dist

from .api import (
    FacetConfig,
    SwiftlyBackward,
    SwiftlyConfig,
    SwiftlyForward,
    make_full_facet_cover,
    make_full_subgrid_cover,
)
from .api_helper import make_facet_device
from .distributed import SwiftlyBackwardSharded, SwiftlyForwardSharded, partition_facets
from .fourier_algorithm import make_subgrid_from_sources

MIB = float(1 << 20)


class OutputSample:
    """The same seeded sample of pixels from each of ``count`` results of one ``shape``,
    gathered on the device as the results appear; at most ``max_bytes`` in all."""

    def __init__(self, shape, count, device, max_pixels=2048, max_bytes=64 * 2**20):
        size = int(numpy.prod(shape))
        n = max(1, min(max_pixels, size, max_bytes // (16 * max(1, count))))
        idx = numpy.sort(numpy.random.default_rng(20261017).choice(size, n, replace=False))
        self.idx = torch.from_numpy(idx).to(device)
        self.rows = {}
        # load the gather kernel now: a first use inside a timed step would pay for it there
        tiny = torch.zeros(1, dtype=torch.complex128, device=device)
        tiny[torch.zeros(1, dtype=torch.int64, device=device)].cpu()

    def __call__(self, i, _config, tensor):
        self.rows[i] = torch.view_as_real(tensor.reshape(-1)[self.idx])

    def array(self):
        """float64 array (results in order, pixels, real / imaginary part)."""
        return numpy.stack([self.rows[i].cpu().numpy() for i in sorted(self.rows)])


class ForwardBenchRunner:
    """Synthetic full-cover forward transform of one parameter set on ``world`` GPUs."""

    # pylint: disable=too-many-instance-attributes
    def __init__(self, params, device, rank=0, world=1, exchange="auto", facet_offsets=None):
        self.exchange = exchange
        self.exchange_used = None
        self.params = dict(params)
        self.device = device
        self.rank = rank
        self.world = world
        self.cfg = SwiftlyConfig(device=device.index, **params)
        self.core = self.cfg.core
        self.facet_cfgs = make_full_facet_cover(self.cfg)
        self.sparse = facet_offsets is not None
        if facet_offsets is not None:  # sparse cover: facets at the given mid-point offsets
            self.facet_cfgs = [FacetConfig(a, b, params["yB_size"]) for a, b in facet_offsets]
        self.sg_cfgs = make_full_subgrid_cover(self.cfg)
        self.owner = partition_facets(self.facet_cfgs, world)
        self.local_idx = [i for i, o in enumerate(self.owner) if o == rank]
        self.yB = params["yB_size"]
        self.yN = params["yN_size"]
        self.xA = params["xA_size"]
        self.xM = params["xM_size"]
        self.m = self.core.xM_yN_size
        F = len(self.local_idx)
        u = self.yB * self.yB  # facet elements
        b = self.yN * self.yB  # prepared facet elements
        # One arena: BF_F[k] at k*b; facet[k] at F*(b-u) + u + k*u.  Stage 1 processes the
        # facets in order; BF_F[k] never reaches a facet that is still unread (see DESIGN.md),
        # so 64 GiB of facets + 128 GiB of BF_F fit in 129 GiB on one GPU at cfg4.
        self.arena = torch.empty(F * b + u, dtype=torch.complex128, device=device)
        self.bf_views = {}
        self.facet_views = {}
        base = F * (b - u) + u
        for k, idx in enumerate(self.local_idx):
            self.bf_views[idx] = self.arena[k * b:(k + 1) * b].view(self.yN, self.yB)
            self.facet_views[idx] = self.arena[base + k * u: base + (k + 1) * u].view(
                self.yB, self.yB)
        self.contributions_per_step = len(self.facet_cfgs) * len(self.sg_cfgs)
        nrows = len({c.off0 for c in self.facet_cfgs})
        ncols = len({s.off0 for s in self.sg_cfgs})
        rows_local = len({self.facet_cfgs[i].off0 for i in self.local_idx})
        # launches of OUR kernels per step on this rank (stage 1, stage 2, axis-1, axis-0)
        owned_sg = len([i for i in range(len(self.sg_cfgs)) if i % world == rank])
        # stage 1 per facet; stage 2 one grouped launch per column (<= 64 facets each);
        # axis 1 one grouped launch per subgrid; axis 0 one launch per owned subgrid
        # (multi-GPU: the axis-1 launch covers a whole batch of world subgrids)
        axis1 = len(self.sg_cfgs) if world == 1 else -(-len(self.sg_cfgs) // world)
        self.launches_per_step = (F + ncols * -(-F // 64) + axis1 + owned_sg)
        self._nrows = nrows
        self._gen = torch.Generator(device=device)

    # ------------------------------------------------------------------ data
    def regenerate_facets(self):
        """Dense standard-normal facets (seed 123456789 + facet index), on the device."""
        for idx in self.local_idx:
            self._gen.manual_seed(123456789 + idx)
            torch.view_as_real(self.facet_views[idx]).normal_(generator=self._gen)

    # ------------------------------------------------------------------ one step
    def _run_forward(self, facet_data, consumer=None):
        if self.world == 1:
            fwd = SwiftlyForward(
                self.cfg, [(fc, facet_data[i]) for i, fc in enumerate(self.facet_cfgs)],
                lru_forward=1, queue_size=4,
                bf_f_buffers=[self.bf_views[i] for i in range(len(self.facet_cfgs))])
            for i, sg in enumerate(self.sg_cfgs):
                task = fwd.get_subgrid_task(sg)
                if consumer is not None:
                    consumer(i, sg, task.tensor)
            return
        fwd = SwiftlyForwardSharded(self.cfg, self.facet_cfgs, facet_data, lru_forward=1,
                                    bf_f_buffers=self.bf_views, exchange=self.exchange)
        self.exchange_used = fwd.exchange
        fwd.get_subgrid_tasks(self.sg_cfgs, consumer=consumer or (lambda *a: None))
        # our kernels actually launched by this rank in the step (+ signal / wait per batch)
        nb = -(-len(self.sg_cfgs) // self.world)
        self.launches_per_step = fwd.launches + (2 * nb if fwd.exchange in ("p2p", "copy") else 0)

    def _barrier(self):
        torch.cuda.synchronize(self.device)
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize(self.device)

    def step(self, timed=True, consumer=None):
        """One complete forward transform; returns its time in ms (max over ranks).
        ``consumer(i, subgrid_config, tensor)`` sees every subgrid this rank finishes."""
        self.regenerate_facets()
        self._barrier()
        start = torch.cuda.Event(enable_timing=True)
        end = torch.cuda.Event(enable_timing=True)
        start.record()
        self._run_forward(self.facet_views, consumer=consumer)
        end.record()
        self._barrier()
        ms = start.elapsed_time(end)
        if self.world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=self.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms if timed else None

    # ------------------------------------------------------------------ output self-check
    def selfcheck(self, n_sources=8, tol=1e-9):
        """Parity of the very path the timed steps ran, at this GPU count.

        The facets are repainted ON THE DEVICE with point sources (zero elsewhere), one more
        complete forward transform runs through the same driver as :meth:`step`, and three
        subgrids owned by this rank (first / middle / last) are compared with the analytic
        DFT of the sources (``make_subgrid_from_sources``, fourier_algorithm.py:267-315).
        Returns the max over ranks of ``max|got - truth| / max|truth|``; raises above ``tol``.
        """
        N = self.params["N"]
        rng = numpy.random.default_rng(20260922)  # same sources on every rank
        if self.sparse:
            # sparse cover: the sources must lie inside covered facets
            sources = []
            for _ in range(n_sources):
                fc = self.facet_cfgs[int(rng.integers(len(self.facet_cfgs)))]
                pos = [(off + int(rng.integers(-self.yB // 2, self.yB // 2)) + N // 2) % N - N // 2
                       for off in (fc.off0, fc.off1)]
                sources.append((float(rng.random()) + 0.5, pos[0], pos[1]))
        else:
            sources = [(float(rng.random()) + 0.5, int(rng.integers(-N // 2, N // 2)),
                        int(rng.integers(-N // 2, N // 2))) for _ in range(n_sources)]
        for idx in self.local_idx:
            make_facet_device(N, self.facet_cfgs[idx], sources, self.device,
                              out=self.facet_views[idx])
        owned = [i for i in range(len(self.sg_cfgs)) if i % self.world == self.rank]
        wanted = sorted({owned[0], owned[len(owned) // 2], owned[-1]}) if owned else []
        kept = {}

        def consumer(i, sg, tensor):
            if i in wanted:
                kept[i] = tensor.clone()

        self._run_forward(self.facet_views, consumer=consumer)
        torch.cuda.synchronize(self.device)
        worst = 0.0
        for i in wanted:
            sg = self.sg_cfgs[i]
            truth = make_subgrid_from_sources(sources, N, sg.size, [sg.off0, sg.off1],
                                              [sg.mask0, sg.mask1])
            got = kept[i].cpu().numpy()
            worst = max(worst, float(numpy.abs(got - truth).max() / numpy.abs(truth).max()))
        checked = len(wanted)
        if self.world > 1:
            t = torch.tensor([worst, float(checked)], dtype=torch.float64, device=self.device)
            dist.all_reduce(t[0:1], op=dist.ReduceOp.MAX)
            dist.all_reduce(t[1:2], op=dist.ReduceOp.SUM)
            worst, checked = float(t[0].item()), int(t[1].item())
        if not worst <= tol:
            raise RuntimeError(f"bench self-check failed: max relative error {worst:.3e} "
                               f"over {checked} subgrids exceeds {tol:g}")
        return {"parity_max_rel_err": worst, "subgrids_checked": checked,
                "against": f"analytic DFT of {n_sources} point sources painted into the facets "
                           "on the device; first / middle / last subgrid owned by every rank; "
                           "max|got - truth| / max|truth|", "tolerance": tol}

    # ------------------------------------------------------------------ per-kernel rooflines
    def _time(self, fn, reps=5):
        fn()
        torch.cuda.synchronize(self.device)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
        evs[0].record()
        for i in range(reps):
            fn()
            evs[i + 1].record()
        torch.cuda.synchronize(self.device)
        return float(numpy.mean([evs[i].elapsed_time(evs[i + 1]) for i in range(reps)]))

    def kernel_rooflines(self, hbm_gbs, step_ms=None):
        """Average duration (CUDA events, this stream) of each kernel of the step, with its
        algorithmic bytes (SURVEY.md section 8d) and the HBM-roofline fraction."""
        core, dev = self.core, self.device
        yB, yN, xA, m = self.yB, self.yN, self.xA, self.m
        fcs = self.facet_cfgs
        idx0 = self.local_idx[0]
        row_members = [i for i in self.local_idx if fcs[i].off0 == fcs[idx0].off0]
        nsrc = len(row_members)
        F = len(self.local_idx)
        ncols = len({s.off0 for s in self.sg_cfgs})
        S = len(self.sg_cfgs)
        rows_local = len({fcs[i].off0 for i in self.local_idx})
        owned_sg = len([i for i in range(S) if i % self.world == self.rank])
        self.regenerate_facets()
        sg = self.sg_cfgs[len(self.sg_cfgs) // 2 + 3]
        out = {}
        t1 = self._time(lambda: core.prepare_facet(
            self.facet_views[idx0], fcs[idx0].off0, axis=0, out=self.bf_views[idx0],
            window_lines=True), 3)
        out["prepare_facet_axis0"] = (t1, 16.0 * (yB * yB + yN * yB), F)
        # make the row's BF_F valid for the following kernels
        for i in row_members:
            core.prepare_facet(self.facet_views[i], fcs[i].off0, axis=0, out=self.bf_views[i],
                               window_lines=True)
        # stage 2 exactly as the step launches it: all local facets of a column in one launch
        for i in self.local_idx:
            core.prepare_facet(self.facet_views[i], fcs[i].off0, axis=0, out=self.bf_views[i],
                               window_lines=True)
        nmbf_all = [torch.empty((m, yN), dtype=torch.complex128, device=dev)
                    for _ in self.local_idx]
        bfs = [self.bf_views[i] for i in self.local_idx]
        off1s = [fcs[i].off1 for i in self.local_idx]
        t2 = self._time(lambda: core.extract_columns(bfs, sg.off0, off1s, outs=nmbf_all,
                                                     prewindowed=True), 3)
        out["extract_columns (Fb.FFT.extract, K2; all local facets of a column)"] = (
            t2, 16.0 * (m * yB + m * yN) * F, ncols)
        nmbf = dict(zip(self.local_idx, nmbf_all))
        nstrips = self._nrows
        strips = torch.empty((nstrips, m, xA), dtype=torch.complex128, device=dev)
        local_rows = sorted({fcs[i].off0 for i in self.local_idx})
        groups = [[(nmbf[i], fcs[i].off1) for i in self.local_idx if fcs[i].off0 == o]
                  for o in local_rows]
        # strips are stored transposed (contribution index contiguous), as in the step
        strips = torch.empty((nstrips, xA, m), dtype=torch.complex128, device=dev).transpose(1, 2)
        if self.world == 1:
            t3 = self._time(lambda: core.sum_finish_axis_grouped(
                groups, strips[:len(groups)], axis=1, subgrid_off=sg.off1))
            out["sum_finish_axis1 (all local facet rows of a subgrid)"] = (
                t3, 16.0 * (F * m * m + len(groups) * m * xA), S)
        else:
            # the step launches the axis-1 kernel for a whole batch: world subgrids of one
            # subgrid column x local facet rows, every group with its own subgrid offset
            batch = [s_ for s_ in self.sg_cfgs if s_.off0 == sg.off0][:self.world]
            bgroups = [g for _ in batch for g in groups]
            boffs = [s_.off1 for s_ in batch for _ in groups]
            bout = torch.empty((len(bgroups), xA, m), dtype=torch.complex128,
                               device=dev).transpose(1, 2)
            t3 = self._time(lambda: core.sum_finish_axis_grouped(
                bgroups, bout, axis=1, subgrid_off=boffs, mask=None))
            out[f"sum_finish_axis1 (batch of {len(batch)} subgrids x local facet rows)"] = (
                t3, 16.0 * len(batch) * (F * m * m + len(groups) * m * xA), -(-S // self.world))
        srcs = groups[0]
        for r in range(nstrips):
            core.sum_finish_axis(srcs, strips[r], axis=1, subgrid_off=sg.off1)
        res = torch.empty((xA, xA), dtype=torch.complex128, device=dev)
        row_offs = sorted({c.off0 for c in fcs})
        srcs0 = [(strips[r], row_offs[r]) for r in range(nstrips)]
        t4 = self._time(lambda: core.sum_finish_axis(srcs0, res, axis=0, subgrid_off=sg.off0))
        out["sum_finish_axis0 (per subgrid)"] = (t4, 16.0 * (nstrips * m * xA + xA * xA), owned_sg)
        # FP64 rate next to every HBM fraction: nominal flops (5 n log2 n per n-point transform)
        # per launch, keyed by the first word of the kernel name
        def fft_flops(n):
            return 5.0 * n * float(numpy.log2(n))

        xM = self.xM
        nominal = {
            "prepare_facet_axis0": yB * fft_flops(yN),
            "extract_columns": F * m * fft_flops(yN),
            "sum_finish_axis1": F * m * fft_flops(m) + len(groups) * m * fft_flops(xM),
            "sum_finish_axis0": xA * (nstrips * fft_flops(m) + fft_flops(xM)),
        }
        if self.world > 1:
            nominal["sum_finish_axis1"] *= len(batch)
        kernels = []
        total = sum(t * n for t, _, n in out.values())
        for name, (t, by, n) in out.items():
            ach = by / (t * 1e-3) / 1e9
            kernels.append({
                "kernel": name, "avg_ms": t, "launches_per_step": n,
                "algorithmic_bytes_per_launch": by, "achieved": ach, "unit": "GB/s",
                "frac": ach / hbm_gbs, "share_of_kernel_time": t * n / total,
                "fp64_nominal_tflops": nominal.get(name.split(" ")[0], 0.0) / (t * 1e-3) / 1e12,
            })
        dom = max(kernels, key=lambda k: k["share_of_kernel_time"])
        dominant = {"bound": "hbm", "achieved": dom["achieved"], "peak": hbm_gbs, "unit": "GB/s",
                    "frac": dom["frac"], "traffic": None, "kernel": dom["kernel"],
                    "avg_ms": dom["avg_ms"],
                    "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"]}
        bmin = None
        if step_ms:
            # B_min of SURVEY.md section 8d, evaluated for this cover
            F_all, S_all = len(fcs), len(self.sg_cfgs)
            per = 16.0 * (F_all * (yB * yB + yN * yB) + ncols * F_all * (m * yB + m * yN)
                          + S_all * F_all * m * m + S_all * xA * xA) / (S_all * F_all)
            by = per * self.contributions_per_step / self.world
            ach = by / (step_ms * 1e-3) / 1e9
            bmin = {"bytes_per_contribution": per, "achieved": ach, "unit": "GB/s",
                    "frac": ach / hbm_gbs, "note": "end-to-end B_min of SURVEY.md section 8d per GPU"}
        return {"kernels": kernels, "dominant": dominant, "bmin": bmin}

    # ------------------------------------------------------------------ end to end (host buffers)
    def e2e(self, steps=1, ring=4, progress=None):
        """Same transform through the public API with HOST buffers: facets start in pinned
        host memory (H2D inside the timed region), every finished subgrid is copied to a
        pinned host buffer (D2H inside the timed region)."""
        yB, xA = self.yB, self.xA
        host = {}
        self.regenerate_facets()
        for n, idx in enumerate(self.local_idx):
            h = torch.empty((yB, yB), dtype=torch.complex128, pin_memory=True)
            h.copy_(self.facet_views[idx])
            host[idx] = h
            if progress is not None and n % 8 == 7:
                progress(f"e2e: pinned {n + 1}/{len(self.local_idx)} host facets")
        slots = [torch.empty((xA, xA), dtype=torch.complex128, pin_memory=True)
                 for _ in range(ring)]
        d2h = torch.cuda.Stream(self.device)
        counter = {"n": 0, "bytes": 0}

        def consumer(i, sg, tensor):
            ev = torch.cuda.Event()
            ev.record()
            d2h.wait_event(ev)
            with torch.cuda.stream(d2h):
                slots[counter["n"] % ring].copy_(tensor, non_blocking=True)
            tensor.record_stream(d2h)
            counter["n"] += 1
            counter["bytes"] += tensor.numel() * 16

        times = []
        for it in range(steps + 1):  # first pass is a warm-up
            counter["n"] = counter["bytes"] = 0
            self._barrier()
            t0 = time.perf_counter()
            self._run_forward(host, consumer=consumer)
            self._barrier()
            dt = time.perf_counter() - t0
            if self.world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=self.device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            if progress is not None:
                progress(f"e2e pass {it}: {dt * 1e3:.1f} ms")
            if it > 0:
                times.append(dt)
        h2d = sum(h.numel() * 16 for h in host.values())
        d2h_bytes = counter["bytes"]
        if self.world > 1:
            t = torch.tensor([h2d, d2h_bytes], dtype=torch.float64, device=self.device)
            dist.all_reduce(t)
            h2d, d2h_bytes = float(t[0].item()), float(t[1].item())
        sec = float(numpy.mean(times))
        return {
            "value": self.contributions_per_step / sec, "unit": "contributions/s",
            "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h_bytes),
            "ms_per_step": sec * 1e3, "steps": steps,
            "path": "SwiftlyForward(host pinned facets) -> get_subgrid_task -> pinned host "
                    "subgrids; wall clock between device synchronisations, max over ranks",
        }


class BackwardBenchRunner:
    """Synthetic full-cover BACKWARD transform (subgrid -> facet, reference ``api.py:327-463``)
    of one parameter set: every subgrid of the cover is folded into every facet.

    One step = ``add_new_subgrid_task`` for all subgrids in cover order (prepare_subgrid,
    extract_from_subgrid(axis 0) per facet row, the fused subgrid_to_facets kernel, the fused
    fold_column kernel whenever a subgrid column is complete) + ``finish()`` (finish_facet
    along axis 0 for every facet).  The subgrid values do not influence the timing: ``n_inputs``
    distinct random subgrids (2 GiB at N=65536, far larger than L2) are fed cyclically, which
    keeps the 64 GiB a full set would need free for the 128 GiB of facet accumulators.
    At N > 1 (:class:`SwiftlyBackwardSharded`) rank ``i % world`` supplies subgrid ``i``.
    """

    def __init__(self, params, device, rank=0, world=1, n_inputs=32):
        self.params = dict(params)
        self.device = device
        self.rank = rank
        self.world = world
        self.cfg = SwiftlyConfig(device=device.index, **params)
        self.core = self.cfg.core
        self.facet_cfgs = make_full_facet_cover(self.cfg)
        self.sg_cfgs = make_full_subgrid_cover(self.cfg)
        self.xA = params["xA_size"]
        gen = torch.Generator(device=device)
        gen.manual_seed(987654321 + rank)
        self.inputs = []
        for _ in range(n_inputs):
            t = torch.empty((self.xA, self.xA), dtype=torch.complex128, device=device)
            torch.view_as_real(t).normal_(generator=gen)
            self.inputs.append(t)
        self.contributions_per_step = len(self.facet_cfgs) * len(self.sg_cfgs)
        self.last_parts = None

    def _barrier(self):
        torch.cuda.synchronize(self.device)
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize(self.device)

    def step(self, timed=True, keep=False):
        """One complete backward transform; returns ms (max over ranks)."""
        self._barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        if self.world == 1:
            bwd = SwiftlyBackward(self.cfg, self.facet_cfgs, lru_backward=1, queue_size=8)
            for i, sg in enumerate(self.sg_cfgs):
                bwd.add_new_subgrid_task(sg, self.inputs[i % len(self.inputs)])
            ev[1].record()
            tasks = bwd.finish()
        else:
            bwd = SwiftlyBackwardSharded(self.cfg, self.facet_cfgs, lru_backward=1, queue_size=8)
            data = [self.inputs[i % len(self.inputs)] if i % self.world == self.rank else None
                    for i in range(len(self.sg_cfgs))]
            bwd.add_subgrid_tasks(self.sg_cfgs, data)
            ev[1].record()
            tasks = list(bwd.finish().values())
        ev[2].record()
        self._barrier()
        ms = ev[0].elapsed_time(ev[2])
        self.last_parts = (ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]))
        if self.world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=self.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        result = tasks if keep else None
        del bwd, tasks
        if not keep:
            torch.cuda.empty_cache()
        return (ms, result) if keep else (ms if timed else None)

    def selfcheck(self, n_pixels=6, tol=5e-8):
        """Parity of the path the timed steps ran: one more complete backward transform in which
        ONE subgrid (middle of the cover) carries ``n_pixels`` non-zero samples and all others
        are zero (they still run through every kernel).  The finished facets must then equal
        the direct DFT of those samples, ``facet[x] = sum_u S[u] exp(-2 pi i u.x / N)`` times the
        facet masks (the inverse of ``make_subgrid_from_sources``, fourier_algorithm.py:267-315;
        SwiFTly reproduces it to its window accuracy: ~3e-9 for a
        single-subgrid delta at W = 13.5625, measured with the reference algorithm).  A 192 x 192 corner block of up
        to three local facets is compared; returns max|got - truth| / max|truth| over ranks."""
        N, xA = self.params["N"], self.xA
        rng = numpy.random.default_rng(424242)
        i0 = len(self.sg_cfgs) // 2 + 5
        sg = self.sg_cfgs[i0]
        pix = [(int(rng.integers(xA)), int(rng.integers(xA)), complex(rng.random() + 0.5,
                                                                      rng.random() - 0.5))
               for _ in range(n_pixels)]
        special = torch.zeros((xA, xA), dtype=torch.complex128, device=self.device)
        for r0, r1, val in pix:
            special[r0, r1] = val
        zero = torch.zeros((xA, xA), dtype=torch.complex128, device=self.device)
        saved = self.inputs
        try:
            class _Feed(list):  # input i of the step: the special subgrid at i0, zeros elsewhere
                def __len__(self):
                    return 1 << 40

                def __getitem__(self, i):
                    return special if i == i0 else zero

            self.inputs = _Feed()
            _, tasks = self.step(timed=True, keep=True)
        finally:
            self.inputs = saved
        owner = partition_facets(self.facet_cfgs, self.world)
        local = [i for i, o in enumerate(owner) if o == self.rank]
        worst, checked, B = 0.0, 0, 192
        for k in sorted({0, len(local) // 2, len(local) - 1}):
            fc = self.facet_cfgs[local[k]]
            got = tasks[k].tensor[:B, :B].cpu().numpy()
            x0 = fc.off0 - fc.size // 2 + numpy.arange(B)
            x1 = fc.off1 - fc.size // 2 + numpy.arange(B)
            truth = numpy.zeros((B, B), dtype=complex)
            for r0, r1, val in pix:
                u0 = sg.off0 - xA // 2 + r0
                u1 = sg.off1 - xA // 2 + r1
                truth += val * numpy.exp(-2j * numpy.pi / N * (u0 * x0[:, None] + u1 * x1[None, :]))
            if fc.mask0 is not None:
                truth *= numpy.asarray(fc.mask0)[:B, None]
            if fc.mask1 is not None:
                truth *= numpy.asarray(fc.mask1)[None, :B]
            worst = max(worst, float(numpy.abs(got - truth).max() / max(numpy.abs(truth).max(), 1e-300)))
            checked += 1
        del tasks
        torch.cuda.empty_cache()
        if self.world > 1:
            t = torch.tensor([worst, float(checked)], dtype=torch.float64, device=self.device)
            dist.all_reduce(t[0:1], op=dist.ReduceOp.MAX)
            dist.all_reduce(t[1:2], op=dist.ReduceOp.SUM)
            worst, checked = float(t[0].item()), int(t[1].item())
        if not worst <= tol:
            raise RuntimeError(f"backward self-check failed: max relative error {worst:.3e} "
                               f"over {checked} facets exceeds {tol:g}")
        return {"parity_max_rel_err": worst, "facets_checked": checked, "tolerance": tol,
                "against": f"direct DFT of {n_pixels} non-zero samples of one subgrid (all other "
                           "subgrids zero) on a 192 x 192 block of first / middle / last local "
                           "facet; max|got - truth| / max|truth|"}

    def kernel_rooflines(self, hbm_gbs):
        """CUDA-event timings of the fused backward kernels in the shapes the step launches,
        with their algorithmic bytes (compulsory reads + read-modify-write of the accumulators)."""
        core, dev = self.core, self.device
        p = self.params
        yB, yN, xA, xM = p["yB_size"], p["yN_size"], p["xA_size"], p["xM_size"]
        m = core.xM_yN_size
        fcs = self.facet_cfgs
        owner = partition_facets(fcs, self.world)
        local = [i for i, o in enumerate(owner) if o == self.rank]
        F = len(local)
        S = len(self.sg_cfgs)
        ncols = len({s.off0 for s in self.sg_cfgs})
        rows = sorted({fcs[i].off0 for i in local})
        sg = self.sg_cfgs[len(self.sg_cfgs) // 2 + 3]

        def timeit(fn, reps=3):
            fn()
            torch.cuda.synchronize(dev)
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
            evs[0].record()
            for i in range(reps):
                fn()
                evs[i + 1].record()
            torch.cuda.synchronize(dev)
            return float(numpy.mean([evs[i].elapsed_time(evs[i + 1]) for i in range(reps)]))

        out = {}
        x = self.inputs[0]
        t = timeit(lambda: core.prepare_subgrid(x, (sg.off0, sg.off1)))
        out["prepare_subgrid (both axes)"] = (t, 16.0 * (xA * xA + 2 * xM * xA + xM * xM), S)
        prepared = core.prepare_subgrid(x, (sg.off0, sg.off1))
        t = timeit(lambda: [core.extract_from_subgrid(prepared, o, axis=0) for o in rows])
        out["extract_from_subgrid axis 0 (all local facet rows)"] = (
            t, 16.0 * len(rows) * (m * xM + m * xM), S)
        blocks = {o: core.extract_from_subgrid(prepared, o, axis=0) for o in rows}
        accs = [torch.zeros((m, yN), dtype=torch.complex128, device=dev) for _ in local]
        t = timeit(lambda: core.subgrid_to_facets(
            [blocks[fcs[i].off0] for i in local], accs, [fcs[i].off1 for i in local], sg.off1))
        out["subgrid_to_facets (extract axis 1 + accumulate, all local facets)"] = (
            t, 16.0 * F * 3 * m * m, S)
        faccs = [torch.zeros((yN, fcs[i].size), dtype=torch.complex128, device=dev)
                 for i in local[:8]]
        n8 = len(faccs)
        t = timeit(lambda: core.fold_column(accs[:n8], faccs, [fcs[i].off1 for i in local[:n8]],
                                            [None] * n8, sg.off0))
        out[f"fold_column (finish axis 1 + add axis 0; timed on {n8} facets, scaled)"] = (
            t * F / n8, 16.0 * F * (m * yN + 2 * m * yB), ncols)
        t = timeit(lambda: core.finish_facet(faccs[0], fcs[local[0]].off0, fcs[local[0]].size, 0))
        out["finish_facet axis 0"] = (t, 16.0 * (yN * yB + yB * yB), F)
        kernels = []
        total = sum(tt * n for tt, _, n in out.values())
        for name, (tt, by, n) in out.items():
            ach = by / (tt * 1e-3) / 1e9
            kernels.append({"kernel": name, "avg_ms": tt, "launches_per_step": n,
                            "algorithmic_bytes_per_launch": by, "achieved": ach, "unit": "GB/s",
                            "frac": ach / hbm_gbs, "share_of_kernel_time": tt * n / total})
        dom = max(kernels, key=lambda k: k["share_of_kernel_time"])
        return {"kernels": kernels,
                "dominant": {"bound": "hbm", "achieved": dom["achieved"], "peak": hbm_gbs,
                             "unit": "GB/s", "frac": dom["frac"], "traffic": None,
                             "kernel": dom["kernel"], "avg_ms": dom["avg_ms"],
                             "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"]}}
