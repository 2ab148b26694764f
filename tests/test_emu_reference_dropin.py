"""
Drop-in at the core-object boundary, checked against outputs recorded from the REAL reference
(``tests/golden/ref_dropin.npz``, written by ``tests/golden/make_golden.py``):

* the task bodies (``api_helper.extract_column``, ``sum_and_finish_subgrid``,
  ``prepare_and_split_subgrid``, ``accumulate_column``, ``accumulate_facet``, ``finish_facet``)
  driven with this repo's core object bound to the host-emulated kernels must give what the
  reference's task bodies gave with its numpy ``SwiftlyCore`` -- the seat
  ``SwiftlyConfig(backend=...)`` fills (reference api.py:137-143);
* the checks of the reference's unit tests (tests/test_core.py: parameters, the 2-D facet <->
  subgrid transforms against the direct DFT, the constant-value 1-D cases) pass with our core
  class and with the ``ska_sdp_func``-shaped adapter (``sdp_func_compat.Swiftly``) in the seat
  of the native library.  The DFT expectations come from this repo's ``fourier_algorithm``,
  which is first pinned to the reference's values stored in the fixture.
"""

import itertools
import os

import numpy
import pytest

from oracle.swiftly_oracle import pad_mid
from ska_sdp_distributed_fourier_transform_b200 import api, api_helper
from ska_sdp_distributed_fourier_transform_b200.fourier_algorithm import (
    make_facet_from_sources, make_subgrid_from_sources)
from tests import parity_cases as pc
from tests.emu_support import emu_core_class

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_dropin.npz")
TEST_PARAMS = dict(W=13.5625, N=1024, yB_size=416, yN_size=512, xA_size=228, xM_size=256)
# point sources (intensity, position 0, position 1) of the reference's 2-D unit tests
F2S_SOURCES = [[(1, 1, 2)], [(1 / 8, 20, 4), (2 / 8, 2, 5), (3 / 8, -5, -4)]]
S2F_SOURCES = [[(1, 0, 0)], [(1, 20, 4)], [(3, -5, 4)]]


@pytest.fixture(scope="module")
def ref():
    return numpy.load(GOLDEN)


def _make(cls, pars):
    return cls(pars["W"], pars["N"], pars["xM_size"], pars["yN_size"])


def test_reference_task_bodies_run_on_our_core(ref):
    W, N, yB, yN, xA, xM = 13.5625, 256, 96, 128, 52, 64
    core = emu_core_class()(W, N, xM, yN)
    facet_cfgs = api_helper.make_full_cover_config(N, yB, api.FacetConfig)
    sg_cfgs = api_helper.make_full_cover_config(N, xA, api.SubgridConfig)
    rng = numpy.random.default_rng(77)
    facets = [pc.rand_c(rng, yB, yB) for _ in facet_cfgs]

    BF_F = [core.prepare_facet(f, fc.off0, axis=0) for f, fc in zip(facets, facet_cfgs)]
    sg = sg_cfgs[7]
    NMBF_BF = [api_helper.extract_column(core, bf, sg.off0, fc.off1)
               for bf, fc in zip(BF_F, facet_cfgs)]
    contribs = [core.extract_from_facet(nb, sg.off1, axis=1) for nb in NMBF_BF]
    subgrid = api_helper.sum_and_finish_subgrid(core, contribs, facet_cfgs, sg)
    pieces = api_helper.prepare_and_split_subgrid(core, subgrid, [sg.off0, sg.off1], facet_cfgs)
    cols = [api_helper.accumulate_column(core, p, None, sg.off1) for p in pieces]
    accs = [api_helper.accumulate_facet(core, c, None, fc, sg.off0)
            for c, fc in zip(cols, facet_cfgs)]
    back = [numpy.asarray(api_helper.finish_facet(core, a, fc)) for a, fc in zip(accs, facet_cfgs)]

    pc.close(numpy.asarray(subgrid), ref["tb_subgrid"], rtol=1e-12,
             what="subgrid through the task bodies")
    assert len(back) == len(ref["tb_back"])
    for a, b, scale in zip(back, ref["tb_back"], ref["tb_back_scale"]):
        assert a.shape == (yB, yB)
        assert numpy.isclose(numpy.abs(a).max(), scale, rtol=1e-11, atol=0)
        err = numpy.abs(a.reshape(-1)[ref["tb_back_idx"]] - b).max()
        assert err <= 1e-11 * scale, f"facet through the task bodies: {err:.3e} vs {scale:.3e}"


def _pin_dft(ref, N, yB, xA, Nx, Ny):
    """This repo's direct DFT gives the reference's expectations; returns the cases."""
    offs_f = [[0, 0], [Ny, Ny], [-Ny, Ny], [0, -Ny]]
    offs_s = [[0, 0], [0, Nx], [Nx, 0], [-Nx, -Nx]]
    idx = ref["dft_sg_idx"]
    got = [make_facet_from_sources(s, N, yB, fo) for s in F2S_SOURCES for fo in offs_f]
    assert numpy.array_equal(numpy.array(got), ref["f2s_facets"])
    got = [make_facet_from_sources(s, N, yB, fo) for s in S2F_SOURCES for fo in offs_f]
    assert numpy.array_equal(numpy.array(got), ref["s2f_facets"])
    for sources, key in ((F2S_SOURCES, "f2s_subgrids"), (S2F_SOURCES, "s2f_subgrids")):
        got = [make_subgrid_from_sources(s, N, xA, so).reshape(-1)[idx]
               for s in sources for so in offs_s]
        numpy.testing.assert_allclose(numpy.array(got), ref[key], rtol=1e-12, atol=1e-15)
    return offs_f, offs_s


def _reference_unit_checks(make, ref, basic=False):
    """The checks of the reference's tests/test_core.py on a core built by ``make(params)``."""
    p = TEST_PARAMS
    N, yB, xA = p["N"], p["yB_size"], p["xA_size"]
    dft = make(p)
    assert (dft.W, dft.N, dft.yN_size, dft.xM_size) == (p["W"], N, p["yN_size"], p["xM_size"])
    assert dft.xM_yN_size == 128
    with pytest.raises(ValueError):
        make(dict(p, N=1050))
    Nx, Ny = dft.subgrid_off_step, dft.facet_off_step
    offs_f, offs_s = _pin_dft(ref, N, yB, xA, Nx, Ny)

    # facet -> subgrid, 2-D, against the direct DFT
    for sources, f_offs in itertools.product(F2S_SOURCES, offs_f):
        facet = make_facet_from_sources(sources, N, yB, f_offs)
        assert numpy.sum(facet) == sum(s[0] for s in sources)
        prepped = dft.prepare_facet(dft.prepare_facet(facet, f_offs[0], axis=0), f_offs[1], axis=1)
        for s_offs in offs_s:
            contrib = dft.extract_from_facet(dft.extract_from_facet(prepped, s_offs[0], axis=0),
                                             s_offs[1], axis=1)
            acc = dft.add_to_subgrid(dft.add_to_subgrid(contrib, f_offs[0], axis=0),
                                     f_offs[1], axis=1)
            subgrid = dft.finish_subgrid(acc, s_offs, xA)
            numpy.testing.assert_array_almost_equal(
                subgrid, make_subgrid_from_sources(sources, N, xA, s_offs), decimal=8)

    # subgrid -> facet, 2-D: the source pixel comes back, everything else stays below it
    for sources, s_offs in itertools.product(S2F_SOURCES, offs_s):
        subgrid = make_subgrid_from_sources(sources, N, xA, s_offs) / xA / xA * N * N
        prepped = dft.prepare_subgrid(subgrid, s_offs)
        for f_offs in offs_f:
            ext = dft.extract_from_subgrid(dft.extract_from_subgrid(prepped, f_offs[0], axis=0),
                                           f_offs[1], axis=1)
            acc = dft.add_to_facet(dft.add_to_facet(ext, s_offs[0], axis=0), s_offs[1], axis=1)
            facet = dft.finish_facet(dft.finish_facet(acc, f_offs[0], yB, axis=0),
                                     f_offs[1], yB, axis=1)
            expected = make_facet_from_sources(sources, N, yB, f_offs)
            numpy.testing.assert_array_almost_equal(
                facet[expected != 0], expected[expected != 0], decimal=11)
            numpy.testing.assert_array_less(facet[expected == 0], numpy.max(expected))

    if not basic:
        return
    # constant-value 1-D cases at odd sizes: a centred point gives a constant subgrid, a
    # constant subgrid gives the value back at the centre of the facet
    xA, yB = xA - 1, yB - 1
    for val, f_off in itertools.product([0, 1, 0.1], numpy.arange(-5 * Ny, 5 * Ny // 2, Ny)):
        facet = numpy.zeros(yB)
        facet[yB // 2 - f_off] = val
        prepped = dft.prepare_facet(facet, f_off, axis=0)
        for s_off in numpy.arange(0, 10 * Nx, Nx):
            acc = dft.add_to_subgrid(dft.extract_from_facet(prepped, s_off, axis=0), f_off, axis=0)
            numpy.testing.assert_array_almost_equal(dft.finish_subgrid(acc, s_off, xA), val / N,
                                                    decimal=15)
    xA, yB = xA + 1, yB + 1
    offs = numpy.arange(-9, 8)
    for val, s_off in itertools.product([0, 1, 0.1], Nx * offs):
        prepped = dft.prepare_subgrid((val / xA) * numpy.ones(xA), s_off)
        for f_off in Ny * offs:
            acc = dft.add_to_facet(dft.extract_from_subgrid(prepped, f_off, axis=0), s_off, axis=0)
            facet = dft.finish_facet(acc, f_off, yB, axis=0)
            numpy.testing.assert_array_almost_equal(facet[yB // 2 - f_off], val, decimal=13)


def test_reference_unit_test_functions_accept_our_core(ref):
    """The reference's unit checks with our core class (emulated kernels) in the seat of its
    numpy ``SwiftlyCore``."""
    cls = emu_core_class()
    _reference_unit_checks(lambda pars: _make(cls, pars), ref)


class _AdapterCore:
    """Core-shaped calls onto the ``ska_sdp_func``-shaped adapter, made the way a caller of the
    native library makes them: every transform runs along the last axis of a 2-D view --
    transposed for axis 0, a single line for 1-D data -- and writes into an array the caller
    allocated (accumulating ones into zeros)."""

    def __init__(self, sw, core):
        self.sw = sw
        self.W, self.N, self.yN_size, self.xM_size = sw.W, sw.N, sw.yN_size, sw.xM_size
        self.xM_yN_size = core.xM_yN_size
        self.subgrid_off_step, self.facet_off_step = core.subgrid_off_step, core.facet_off_step

    @staticmethod
    def _view(a, axis):
        if a.ndim == 1:
            return a[None, :]
        return a.T if axis == 0 else a

    def _along(self, name, data, size, off, axis):
        data = numpy.asarray(data, dtype=complex)
        shape = list(data.shape)
        shape[axis] = size
        out = numpy.zeros(shape, dtype=complex)
        getattr(self.sw, name)(self._view(data, axis), self._view(out, axis), off)
        return out

    def prepare_facet(self, facet, off, axis):
        return self._along("prepare_facet", facet, self.yN_size, off, axis)

    def extract_from_facet(self, prep, off, axis):
        return self._along("extract_from_facet", prep, self.xM_yN_size, off, axis)

    def add_to_subgrid(self, contrib, off, axis):
        return self._along("add_to_subgrid", contrib, self.xM_size, off, axis)

    def finish_subgrid(self, acc, offs, size):
        offs = numpy.atleast_1d(offs)
        for axis, off in enumerate(offs):
            acc = self._along("finish_subgrid", acc, size, off, axis)
        return acc

    def prepare_subgrid(self, subgrid, offs):
        offs = numpy.atleast_1d(offs)
        padded = numpy.asarray(subgrid, dtype=complex)
        for axis in range(padded.ndim):
            padded = pad_mid(padded, self.xM_size, axis)
        padded = numpy.ascontiguousarray(padded)
        for axis, off in enumerate(offs):
            view = self._view(padded, axis)
            self.sw.prepare_subgrid_inplace(view, int(off))
        return padded

    def extract_from_subgrid(self, psg, off, axis):
        return self._along("extract_from_subgrid", psg, self.xM_yN_size, off, axis)

    def add_to_facet(self, contrib, off, axis):
        return self._along("add_to_facet", contrib, self.yN_size, off, axis)

    def finish_facet(self, acc, off, size, axis):
        return self._along("finish_facet", acc, size, off, axis)


def test_unmodified_reference_native_backend_runs_on_our_library(ref):
    """The reference's unit checks -- 2-D transforms through transposed strided views and the
    constant-value 1-D cases at odd sizes included -- with the ``ska_sdp_func``-shaped adapter
    (emulated kernels here) in the seat of the native library."""
    from ska_sdp_distributed_fourier_transform_b200 import _lib, sdp_func_compat

    cls = emu_core_class()
    lib = cls(13.5625, 256, 64, 128)._lib

    class EmuSwiftly(sdp_func_compat.Swiftly):
        def __init__(self, N, yN_size, xM_size, W):
            real = _lib.load
            _lib.load = lambda path=None: lib
            try:
                super().__init__(N, yN_size, xM_size, W)
            finally:
                _lib.load = real

    def make(pars):
        sw = EmuSwiftly(pars["N"], pars["yN_size"], pars["xM_size"], pars["W"])
        return _AdapterCore(sw, _make(cls, pars))

    _reference_unit_checks(make, ref, basic=True)
