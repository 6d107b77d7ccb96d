"""CPU-only checks of device output (bsg_*_device, `out=` / `device=`): the entry points exist and refuse to run without a
GPU, the Python side rejects unusable buffers before the library sees them, and CountSignals over a torch buffer gives
the shapes and element order of the numpy one."""
import ctypes as C
import os

import numpy as np
import pytest

import bamsignals_b200 as B
from bamsignals_b200 import api


class DeviceArray:
    """A stand-in for a device array: only __cuda_array_interface__ (version 3)."""

    def __init__(self, n, typestr="<i4", strides=None, ptr=0x7f0000000000, shape=None, stream=None):
        self.__cuda_array_interface__ = dict(shape=shape or (n,), typestr=typestr, data=(ptr, False), strides=strides,
                                             version=3)
        if stream is not None:
            self.__cuda_array_interface__["stream"] = stream


def no_gpu():
    return B.lib().bsg_device_count() == 0


def test_device_entry_points_exported():
    L = B.lib()
    for s in ("bsg_pileup_device", "bsg_coverage_device", "bsg_pileup_staged_device", "bsg_coverage_staged_device"):
        assert hasattr(L, s)


def test_device_entry_points_need_a_gpu(fixture_bam):
    if not no_gpu():
        pytest.skip("a GPU is present")
    gr = B.GRanges(["chr1", "chr2"], [1, 100], [10, 20], ["+", "-"])
    for call in (lambda: B.pileup_core(fixture_bam, gr, None, binsize=1, out=DeviceArray(30)),
                 lambda: B.pileup_core(fixture_bam, gr, None, binsize=-1, ss=True, out=DeviceArray(4)),
                 lambda: B.coverage_core(fixture_bam, gr, None, out=DeviceArray(30))):
        with pytest.raises(B.BamsignalsError, match="no CUDA device") as e:
            call()
        assert e.value.code == -6
    off = np.zeros(1, dtype=np.int64)
    assert B.lib().bsg_pileup_staged_device(None, None, 0, 1, 0, 0, 0, -1, 0, None, api._p(off, C.c_int64), None) == -8
    assert B.lib().bsg_coverage_staged_device(None, None, 0, 0, -1, 0, None, api._p(off, C.c_int64), None) == -8


def test_python_rejects_unusable_buffers(fixture_bam):
    gr = B.GRanges(["chr1", "chr2"], [1, 100], [10, 20], ["+", "-"])
    cases = [(np.zeros(30, np.int32), TypeError),                           # host memory has no device interface
             (DeviceArray(30, typestr="<i8"), TypeError),
             (DeviceArray(30, strides=(8,)), ValueError),
             (DeviceArray(29), ValueError),
             (DeviceArray(30, shape=(15, 2)), ValueError)]
    torch = pytest.importorskip("torch")
    cases += [(torch.zeros(30, dtype=torch.int32), TypeError),              # a CPU tensor
              (torch.zeros(30, dtype=torch.int64), TypeError)]
    for buf, err in cases:
        with pytest.raises(err):
            B.pileup_core(fixture_bam, gr, None, binsize=1, out=buf)
        with pytest.raises(err):
            B.coverage_core(fixture_bam, gr, None, out=buf)
    with pytest.raises(TypeError):
        B.bamCoverage(fixture_bam, gr, device="cpu")


def test_device_buffer_checks_in_order():
    """dtype / shape / contiguity / length of any __cuda_array_interface__ object; its stream entry is passed on."""
    assert api.device_buffer(DeviceArray(10, ptr=4096), 10) == (4096, 0)
    assert api.device_buffer(DeviceArray(10, ptr=4096, stream=1), 8) == (4096, 1)
    assert api.device_buffer(DeviceArray(1, strides=(8,)), 1)[0] == 0x7f0000000000       # one element: any stride
    with pytest.raises(ValueError, match="needs 11"):
        api.device_buffer(DeviceArray(10), 11)
    with pytest.raises(ValueError, match="C-contiguous"):
        api.device_buffer(DeviceArray(10, strides=(-4,)), 10)


def _ref_views(flat, off, ss):
    out = []
    for i in range(len(off) - 1):
        v = flat[off[i]:off[i + 1]]
        out.append(v.reshape((2, -1), order="F") if ss else v)
    return out


@pytest.mark.parametrize("ss", [False, True])
def test_countsignals_over_a_torch_buffer(ss):
    torch = pytest.importorskip("torch")
    w = np.array([3, 0, 5, 2, 1], dtype=np.int32)
    off = api.output_layout(w, 1, ss)
    flat = (np.arange(off[-1], dtype=np.int32) * 7) % 101
    a = B.CountSignals(None, ss, flat=flat, offsets=off)
    t = B.CountSignals(None, ss, flat=torch.from_numpy(flat.copy()), offsets=off)
    assert len(a) == len(t) == len(w) and np.array_equal(a.width(), t.width())
    ref = _ref_views(flat, off, ss)
    for i in range(len(w)):
        assert isinstance(t[i], torch.Tensor)
        assert tuple(t[i].shape) == a[i].shape == ref[i].shape
        assert np.array_equal(t[i].numpy(), a[i]) and np.array_equal(a[i], ref[i])
    for x, y in zip(t.as_list(), a.as_list()):
        assert tuple(x.shape) == y.shape and np.array_equal(x.numpy(), y)
    sub_t, sub_a = t[[4, 0, 2]], a[[4, 0, 2]]
    for x, y in zip(sub_t.as_list(), sub_a.as_list()):
        assert tuple(x.shape) == y.shape and np.array_equal(x.numpy(), y)
    with pytest.raises(ValueError):
        t.alignSignals()                                    # widths differ


@pytest.mark.parametrize("ss", [False, True])
@pytest.mark.parametrize("width", [4, 0])
def test_align_signals_over_a_torch_buffer(ss, width):
    torch = pytest.importorskip("torch")
    w = np.full(3, width, dtype=np.int32)
    off = api.output_layout(w, 1, ss)
    flat = np.arange(off[-1], dtype=np.int32)
    a = B.CountSignals(None, ss, flat=flat, offsets=off)
    t = B.CountSignals(None, ss, flat=torch.from_numpy(flat.copy()), offsets=off)
    want = np.stack(_ref_views(flat, off, ss), axis=-1)     # simplify2array: [w, R] or [2, w, R]
    for got in (t.alignSignals(), t[[0, 1, 2]].alignSignals()):   # one reshape of the flat buffer; torch.stack of views
        assert isinstance(got, torch.Tensor)
        assert tuple(got.shape) == want.shape and np.array_equal(got.numpy(), want)
    for got in (a.alignSignals(), a[[0, 1, 2]].alignSignals()):
        assert got.shape == want.shape and np.array_equal(got, want)


def test_package_imports_without_torch():
    import subprocess
    import sys
    code = ("import sys; sys.modules['torch'] = None; import bamsignals_b200 as B; import numpy as np; "
            "from bamsignals_b200 import api; "
            "cs = B.CountSignals(None, True, flat=np.arange(8, dtype=np.int32), offsets=np.array([0, 4, 8])); "
            "assert cs.alignSignals().shape == (2, 2, 2)")
    subprocess.check_call([sys.executable, "-c", code], cwd=api.os.path.dirname(api.os.path.dirname(api.__file__)))


def test_empty_align_signals_stays_a_tensor():
    torch = pytest.importorskip("torch")
    t = B.CountSignals(None, False, flat=torch.zeros(0, dtype=torch.int32), offsets=np.zeros(1, np.int64))
    got = t.alignSignals()
    assert isinstance(got, torch.Tensor) and tuple(got.shape) == (0,) and got.dtype == torch.int32


def test_device_must_be_cuda_before_anything_is_allocated(fixture_bam):
    pytest.importorskip("torch")
    gr = B.GRanges(["chr1"], [1], [10])
    with pytest.raises(TypeError, match="must be a CUDA device"):
        B.bamProfile(fixture_bam, gr, device="cpu")


# ---- the tile kernels' index ranges for a destination of any 16-byte phase ------------------------------------------
# k_profile / k_profile_agg / k_coverage place their shared buffer at the phase of the destination ADDRESS, so that the
# body of a tile moves as 128-bit shared loads and 128-bit streaming stores even when the caller's buffer (bsg_*_device)
# is only 4-byte aligned.  Restated here from kernels.cu: every shared access must stay inside the dynamic shared memory
# the launcher sizes, every vector access must be 16-byte aligned, and the global stores must cover the tile's ints
# exactly once and nothing else.

def kernels_src():
    return open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bamsignals_b200", "csrc",
                             "kernels.cu")).read()


def test_kernel_source_matches_the_restatement():
    src = kernels_src()
    assert src.count("out_phase(out + off)") == 3 and "off & 3" not in src
    assert "size_t(max_tile_ints + 4) * sizeof(int32_t)" in src          # launch_profile: both profile kernels
    assert "size_t(max_tile_ints + 8) * sizeof(int32_t)" in src          # launch_coverage
    assert "int32_t* dst = out + off - ph;" in src


def copy_out_accesses(a, ph, n):
    """copy_out(dst = int address a, sm = smem + ph, n): (shared ints read, global ints written, vector accesses)."""
    head = min(n, (4 - (a & 3)) & 3)
    body = (n - head) >> 2
    sh, gl, vec = [], [], []
    for t in range(head):
        sh.append(ph + t); gl.append(a + t)
    for k in range(body):
        s0, g0 = ph + head + 4 * k, a + head + 4 * k
        vec += [s0, g0]
        sh += range(s0, s0 + 4); gl += range(g0, g0 + 4)
    for t in range(head + 4 * body, n):
        sh.append(ph + t); gl.append(a + t)
    return sh, gl, vec


def coverage_accesses(a, ln):
    """k_coverage for a tile of ln ints at int address a: (shared ints touched, global ints written, vector accesses)."""
    ph = a & 3
    total = ph + ln
    nquads = (total + 3) >> 2
    sh = list(range(4 * nquads)) + [ph + j for j in range(ln)]         # zero-fill / scan in quads; d[0..ln) = smem[ph..]
    dst = a - ph
    gl, vec = [], [dst]
    for q in range(nquads):
        j = 4 * q
        if j >= ph and j + 4 <= total:
            vec.append(dst + j); gl += range(dst + j, dst + j + 4)
        else:
            gl += [dst + j + i for i in range(4) if ph <= j + i < total]
    return sh, gl, vec


TILE_LENS = list(range(0, 70)) + [1000, 4093, 4094, 4095, 4096, 8189, 8190, 8191, 8192]


@pytest.mark.parametrize("base", [0, 1, 2, 3, 1 << 20])
def test_tile_kernels_stay_in_bounds_at_every_phase(base):
    """base: int address of the caller's out[0]; off: the tile's offset in it (cudaMalloc'd smem is 16-byte aligned)."""
    for ln in TILE_LENS:
        for off in (0, 1, 2, 3, 7, 1234):
            a = base + off
            ph = a & 3
            # profile (both kernels): nout <= max_tile_ints; worst case: this tile is the largest one
            sh, gl, vec = copy_out_accesses(a, ph, ln)
            assert all(0 <= i < ln + 4 for i in sh), (a, ln)
            assert sorted(gl) == list(range(a, a + ln)), (a, ln)
            assert all(v % 4 == 0 for v in vec), (a, ln)
            sh, gl, vec = coverage_accesses(a, ln)
            assert all(0 <= i < ln + 8 for i in sh), (a, ln)
            assert sorted(gl) == list(range(a, a + ln)), (a, ln)
            assert all(v % 4 == 0 for v in vec), (a, ln)
