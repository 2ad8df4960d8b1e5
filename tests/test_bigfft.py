"""The large-FFT Welch paths (N >= 16384: four-step and radix-16) against the oracle: each
scenario of tests/bigfft_suite.py once on the CPU emulation build of the engine sources and
once, marked gpu, on the sm_100a library on the B200."""
import pytest

from tests import bigfft_suite as bs


@pytest.mark.parametrize("name", sorted(bs.PINNED))
def test_pinned_dc_case(emu_engine, name):
    bs.pinned_case(emu_engine, name)


@pytest.mark.parametrize("N", bs.LARGE)
def test_dc_offsets(emu_engine, N):
    bs.dc_offsets(emu_engine, N)


@pytest.mark.parametrize("N", bs.LARGE)
def test_per_frame_dc(emu_engine, N):
    bs.per_frame_dc(emu_engine, N)


@pytest.mark.parametrize("N", bs.LARGE)
def test_crop_and_zoom(emu_engine, N):
    bs.crop_and_zoom(emu_engine, N)


@pytest.mark.parametrize("N", bs.LARGE)
def test_fp64_fp32_boundary(emu_engine, N):
    bs.fp64_fp32_boundary(emu_engine, N)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_large(emu_engine, seed):
    bs.random_large(emu_engine, seed, 8)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(bs.PINNED))
def test_pinned_dc_case_gpu(gpu_engine, name):
    bs.pinned_case(gpu_engine, name)


@pytest.mark.gpu
@pytest.mark.parametrize("N", bs.LARGE)
def test_dc_offsets_gpu(gpu_engine, N):
    bs.dc_offsets(gpu_engine, N)


@pytest.mark.gpu
@pytest.mark.parametrize("N", bs.LARGE)
def test_per_frame_dc_gpu(gpu_engine, N):
    bs.per_frame_dc(gpu_engine, N)


@pytest.mark.gpu
@pytest.mark.parametrize("N", bs.LARGE)
def test_crop_and_zoom_gpu(gpu_engine, N):
    bs.crop_and_zoom(gpu_engine, N)


@pytest.mark.gpu
@pytest.mark.parametrize("N", bs.LARGE)
def test_fp64_fp32_boundary_gpu(gpu_engine, N):
    bs.fp64_fp32_boundary(gpu_engine, N)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [11, 12, 13, 14])
def test_random_large_gpu(gpu_engine, seed):
    bs.random_large(gpu_engine, seed, 10)
