#!/usr/bin/env python
"""
Generate golden fixtures from the REAL reference implementation.

Run where a checkout of the reference (ska-sdp-exec-swiftly) exists:

    python tests/golden/make_golden.py <reference checkout>/src [fixture ...]

It imports the unmodified reference package ``ska_sdp_exec_swiftly`` (numpy
backend ``SwiftlyCore`` and the ``api_helper`` task bodies) from the given
source directory -- with tiny stub modules standing in for the
uninstallable ``dask`` / ``distributed`` / ``ska_sdp_func`` imports, exactly as
described in SURVEY.md Appendix A -- runs it on seeded inputs and stores inputs
and outputs as ``tests/golden/*.npz`` (all of them, or only the named fixtures:
``1d``, ``2d``, ``windows``, ``dropin``).  Those files pin the oracle
(``tests/test_oracle.py``) and the kernels (``tests/test_emu_reference_dropin.py``).
"""

import os
import sys
import types

import numpy

HERE = os.path.dirname(os.path.abspath(__file__))


def _install_stubs():
    """Stub the reference's uninstallable imports (never used by the numpy path)."""

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    class _Unavailable:  # pylint: disable=too-few-public-methods
        def __init__(self, *a, **k):
            raise ImportError("stub: not installed in this container")

    def _delayed(*a, **k):
        raise ImportError("stub: dask not installed")

    func = mod("ska_sdp_func")
    ft = mod("ska_sdp_func.fourier_transforms")
    sw = mod("ska_sdp_func.fourier_transforms.swiftly", Swiftly=_Unavailable)
    func.fourier_transforms = ft
    ft.swiftly = sw
    dask = mod("dask", delayed=_delayed)
    dask.array = mod("dask.array")
    dask.distributed = mod("dask.distributed")
    mod("distributed", Client=_Unavailable)


def import_reference(ref_src):
    _install_stubs()
    if ref_src not in sys.path:
        sys.path.insert(0, ref_src)
    # pylint: disable=import-outside-toplevel
    from ska_sdp_exec_swiftly import api, api_helper
    from ska_sdp_exec_swiftly.fourier_transform import core, fourier_algorithm

    return api, api_helper, core, fourier_algorithm


def rand_c(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


TEST_PARAMS = dict(W=13.5625, N=1024, yB_size=416, yN_size=512, xA_size=228, xM_size=256)
SMALL_PARAMS = dict(W=13.5625, N=256, yB_size=96, yN_size=128, xA_size=52, xM_size=64)


def golden_1d(core_mod):
    """All eight primitives in 1-D at the reference's TEST_PARAMS."""
    p = TEST_PARAMS
    core = core_mod.SwiftlyCore(p["W"], p["N"], p["xM_size"], p["yN_size"])
    rng = numpy.random.default_rng(20240901)
    Nx, Ny = core.subgrid_off_step, core.facet_off_step
    out = {"Fb": core._Fb, "Fn": core._Fn}
    cases = []
    idx = 0
    for yB in (p["yB_size"], p["yB_size"] - 1):
        for xA in (p["xA_size"], p["xA_size"] - 1):
            for facet_off, sg_off in ((0, 0), (3 * Ny, 5 * Nx), (-7 * Ny, -2 * Nx), (p["N"], p["N"] + Nx)):
                facet = rand_c(rng, yB)
                prep = core.prepare_facet(facet, facet_off, axis=0)
                contrib = core.extract_from_facet(prep, sg_off, axis=0)
                acc = core.add_to_subgrid(contrib, facet_off, axis=0)
                sg = core.finish_subgrid(acc, sg_off, xA)
                subgrid = rand_c(rng, xA)
                psg = core.prepare_subgrid(subgrid, sg_off)
                ext = core.extract_from_subgrid(psg, facet_off, axis=0)
                accf = core.add_to_facet(ext, sg_off, axis=0)
                fin = core.finish_facet(accf, facet_off, yB, axis=0)
                for k, v in dict(
                    facet=facet, prep=prep, contrib=contrib, acc=acc, sg=sg,
                    subgrid=subgrid, psg=psg, ext=ext, accf=accf, fin=fin,
                ).items():
                    out[f"c{idx}_{k}"] = v
                cases.append((yB, xA, facet_off, sg_off))
                idx += 1
    out["cases"] = numpy.array(cases, dtype=numpy.int64)
    out["params"] = numpy.array([p["W"], p["N"], p["xM_size"], p["yN_size"]])
    numpy.savez_compressed(os.path.join(HERE, "ref_1d_n1024.npz"), **out)
    print("ref_1d_n1024.npz", idx, "cases")


def golden_2d(api, api_helper, core_mod):
    """2-D primitives, both axes, plus a full forward+backward through the
    reference's own task bodies, at a small valid parameter set."""
    p = SMALL_PARAMS
    core = core_mod.SwiftlyCore(p["W"], p["N"], p["xM_size"], p["yN_size"])
    rng = numpy.random.default_rng(20240902)
    Nx, Ny = core.subgrid_off_step, core.facet_off_step
    yB, xA, m = p["yB_size"], p["xA_size"], core.xM_yN_size
    out = {"Fb": core._Fb, "Fn": core._Fn,
           "params": numpy.array([p["W"], p["N"], p["xM_size"], p["yN_size"], yB, xA])}

    # primitive by primitive, axis by axis (odd sizes along the active axis)
    f_off, s_off = 5 * Ny, -3 * Nx
    for axis in (0, 1):
        shape = [19, 19]
        shape[axis] = yB - 1
        facet = rand_c(rng, *shape)
        prep = core.prepare_facet(facet, f_off, axis=axis)
        contrib = core.extract_from_facet(prep, s_off, axis=axis)
        acc0 = rand_c(rng, *[p["xM_size"] if a == axis else 19 for a in (0, 1)])
        acc = core.add_to_subgrid(contrib, f_off, axis=axis, out=acc0.copy())
        fin = core.finish_facet(prep, f_off, yB - 1, axis=axis)
        ext = core.extract_from_subgrid(acc, f_off, axis=axis)
        accf0 = rand_c(rng, *prep.shape)
        accf = core.add_to_facet(ext, s_off, axis=axis, out=accf0.copy())
        for k, v in dict(facet=facet, prep=prep, contrib=contrib, acc0=acc0, acc=acc,
                         fin=fin, ext=ext, accf0=accf0, accf=accf).items():
            out[f"ax{axis}_{k}"] = v
    out["prim_offs"] = numpy.array([f_off, s_off])
    summed = rand_c(rng, p["xM_size"], p["xM_size"])
    out["fs_in"] = summed
    out["fs_out"] = core.finish_subgrid(summed, [2 * Nx, -Nx], xA - 1)
    sgin = rand_c(rng, xA - 1, xA - 1)
    out["ps_in"] = sgin
    out["ps_out"] = core.prepare_subgrid(sgin, (2 * Nx, -Nx))

    # full forward + backward with the reference's task bodies (serial, no dask)
    class Cfg:  # pylint: disable=too-few-public-methods
        N = p["N"]

    facet_cfgs = api_helper.make_full_cover_config(p["N"], yB, api.FacetConfig)
    sg_cfgs = api_helper.make_full_cover_config(p["N"], xA, api.SubgridConfig)
    facets = [rand_c(rng, yB, yB) * fc.mask0[:, None] * fc.mask1[None, :] for fc in facet_cfgs]
    BF_F = [core.prepare_facet(f, fc.off0, axis=0) for f, fc in zip(facets, facet_cfgs)]
    subgrids = []
    cur = None
    NMBF_BF = None
    # backward state
    MNAF_BMNAF = [None] * len(facet_cfgs)
    NAF_MNAF = [None] * len(facet_cfgs)
    for sg in sg_cfgs:
        if sg.off0 != cur:
            if cur is not None:
                MNAF_BMNAF = [
                    api_helper.accumulate_facet(core, NAF_MNAF[j], MNAF_BMNAF[j], fc, cur)
                    for j, fc in enumerate(facet_cfgs)
                ]
                NAF_MNAF = [None] * len(facet_cfgs)
            cur = sg.off0
            NMBF_BF = [
                api_helper.extract_column(core, bf, sg.off0, fc.off1)
                for bf, fc in zip(BF_F, facet_cfgs)
            ]
        contribs = [core.extract_from_facet(nb, sg.off1, axis=1) for nb in NMBF_BF]
        res = api_helper.sum_and_finish_subgrid(core, contribs, facet_cfgs, sg)
        subgrids.append(res)
        naf = api_helper.prepare_and_split_subgrid(core, res, [sg.off0, sg.off1], facet_cfgs)
        NAF_MNAF = [
            api_helper.accumulate_column(core, naf[j], NAF_MNAF[j], sg.off1)
            for j in range(len(facet_cfgs))
        ]
    MNAF_BMNAF = [
        api_helper.accumulate_facet(core, NAF_MNAF[j], MNAF_BMNAF[j], fc, cur)
        for j, fc in enumerate(facet_cfgs)
    ]
    back = [api_helper.finish_facet(core, MNAF_BMNAF[j], fc) for j, fc in enumerate(facet_cfgs)]
    out["facet_offs"] = numpy.array([[fc.off0, fc.off1] for fc in facet_cfgs])
    out["sg_offs"] = numpy.array([[sg.off0, sg.off1] for sg in sg_cfgs])
    out["facet_mask0"] = numpy.array([fc.mask0 for fc in facet_cfgs])
    out["facet_mask1"] = numpy.array([fc.mask1 for fc in facet_cfgs])
    out["sg_mask0"] = numpy.array([sg.mask0 for sg in sg_cfgs])
    out["sg_mask1"] = numpy.array([sg.mask1 for sg in sg_cfgs])
    out["facets"] = numpy.array(facets)
    out["subgrids"] = numpy.array(subgrids)
    out["back_facets"] = numpy.array(back)
    out["NMBF_BF_last"] = numpy.array(NMBF_BF)
    out["BF_F0"] = BF_F[0]
    numpy.savez_compressed(os.path.join(HERE, "ref_2d_n256.npz"), **out)
    print("ref_2d_n256.npz", len(facet_cfgs), "facets", len(sg_cfgs), "subgrids")


def golden_windows(core_mod):
    """PSWF-derived Fb / Fn tables for the BASELINE parameter sets (scipy pins them)."""
    out = {}
    for name, (W, N, xM, yN) in {
        "cfg1": (13.5625, 1024, 256, 512),
        "cfg2": (13.5625, 8192, 2048, 4096),
        "cfg3": (13.5625, 32768, 4096, 8192),
        "cfg4": (13.5625, 65536, 4096, 16384),
    }.items():
        core = core_mod.SwiftlyCore(W, N, xM, yN)
        # store sub-sampled tables (every 16th sample) plus a checksum of the whole
        out[f"{name}_Fb_s"] = core._Fb[::16]
        out[f"{name}_Fn_s"] = core._Fn[::16]
        out[f"{name}_sums"] = numpy.array([core._Fb.sum(), core._Fn.sum(),
                                           (core._Fb ** 2).sum(), (core._Fn ** 2).sum()])
    numpy.savez_compressed(os.path.join(HERE, "ref_windows.npz"), **out)
    print("ref_windows.npz")


def golden_dropin(api, api_helper, core_mod, fourier_algorithm):
    """What tests/test_emu_reference_dropin.py compares against.

    * A forward + backward pass through the reference's task bodies at SMALL_PARAMS, facets
      from ``default_rng(77)``, subgrid 7 of the cover: the subgrid, and the backward facets
      at DROPIN_SAMPLES seeded pixels together with each facet's largest magnitude.
    * The direct-DFT expectations of the reference's 2-D unit tests at TEST_PARAMS: the point
      source facets (dense; they compress to almost nothing) and the subgrids at
      DROPIN_SAMPLES seeded pixels.
    """
    p = SMALL_PARAMS
    core = core_mod.SwiftlyCore(p["W"], p["N"], p["xM_size"], p["yN_size"])
    yB, xA = p["yB_size"], p["xA_size"]
    facet_cfgs = api_helper.make_full_cover_config(p["N"], yB, api.FacetConfig)
    sg_cfgs = api_helper.make_full_cover_config(p["N"], xA, api.SubgridConfig)
    rng = numpy.random.default_rng(77)
    facets = [rand_c(rng, yB, yB) for _ in facet_cfgs]
    BF_F = [core.prepare_facet(f, fc.off0, axis=0) for f, fc in zip(facets, facet_cfgs)]
    sg = sg_cfgs[7]
    NMBF_BF = [api_helper.extract_column(core, bf, sg.off0, fc.off1)
               for bf, fc in zip(BF_F, facet_cfgs)]
    contribs = [core.extract_from_facet(nb, sg.off1, axis=1) for nb in NMBF_BF]
    subgrid = api_helper.sum_and_finish_subgrid(core, contribs, facet_cfgs, sg)
    pieces = api_helper.prepare_and_split_subgrid(core, subgrid, [sg.off0, sg.off1], facet_cfgs)
    cols = [api_helper.accumulate_column(core, pc, None, sg.off1) for pc in pieces]
    accs = [api_helper.accumulate_facet(core, c, None, fc, sg.off0)
            for c, fc in zip(cols, facet_cfgs)]
    back = numpy.array([api_helper.finish_facet(core, a, fc) for a, fc in zip(accs, facet_cfgs)])
    pick = numpy.random.default_rng(78)
    back_idx = numpy.sort(pick.choice(yB * yB, DROPIN_SAMPLES, replace=False))
    out = {"tb_subgrid": subgrid, "tb_back_idx": back_idx,
           "tb_back": back.reshape(len(back), -1)[:, back_idx],
           "tb_back_scale": numpy.abs(back).max(axis=(1, 2))}

    t = TEST_PARAMS
    N, yB, xA = t["N"], t["yB_size"], t["xA_size"]
    tcore = core_mod.SwiftlyCore(t["W"], N, t["xM_size"], t["yN_size"])
    Nx, Ny = tcore.subgrid_off_step, tcore.facet_off_step
    sg_idx = numpy.sort(pick.choice(xA * xA, DROPIN_SAMPLES, replace=False))
    out["dft_sg_idx"] = sg_idx
    # facet -> subgrid: point sources in facets, direct DFT of the subgrids
    f2s_sources, s2f_sources = dropin_sources()
    offs_f = [[0, 0], [Ny, Ny], [-Ny, Ny], [0, -Ny]]
    offs_s = [[0, 0], [0, Nx], [Nx, 0], [-Nx, -Nx]]
    out["f2s_facets"] = numpy.array([
        fourier_algorithm.make_facet_from_sources(src, N, yB, fo)
        for src in f2s_sources for fo in offs_f])
    out["f2s_subgrids"] = numpy.array([
        fourier_algorithm.make_subgrid_from_sources(src, N, xA, so).reshape(-1)[sg_idx]
        for src in f2s_sources for so in offs_s])
    # subgrid -> facet: DFT subgrids in, point sources in the facets expected
    out["s2f_subgrids"] = numpy.array([
        fourier_algorithm.make_subgrid_from_sources(src, N, xA, so).reshape(-1)[sg_idx]
        for src in s2f_sources for so in offs_s])
    out["s2f_facets"] = numpy.array([
        fourier_algorithm.make_facet_from_sources(src, N, yB, fo)
        for src in s2f_sources for fo in offs_f])
    numpy.savez_compressed(os.path.join(HERE, "ref_dropin.npz"), **out)
    print("ref_dropin.npz")


DROPIN_SAMPLES = 2048


def dropin_sources():
    """Point sources (intensity, position 0, position 1) of the reference's 2-D unit tests:
    facet -> subgrid, subgrid -> facet."""
    return ([[(1, 1, 2)], [(1 / 8, 20, 4), (2 / 8, 2, 5), (3 / 8, -5, -4)]],
            [[(1, 0, 0)], [(1, 20, 4)], [(3, -5, 4)]])


def main(ref_src, names=()):
    api, api_helper, core_mod, fourier_algorithm = import_reference(ref_src)
    makers = {
        "1d": lambda: golden_1d(core_mod),
        "2d": lambda: golden_2d(api, api_helper, core_mod),
        "windows": lambda: golden_windows(core_mod),
        "dropin": lambda: golden_dropin(api, api_helper, core_mod, fourier_algorithm),
    }
    for name in names or makers:
        makers[name]()


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2:])
