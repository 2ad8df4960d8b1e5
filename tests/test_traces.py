"""Max-hold / min-hold / average traces and peak markers (DESIGN 3.8): each scenario of
tests/traces_suite.py once on the CPU emulation build of the engine sources and once,
marked gpu, on the sm_100a library on the B200."""
import pytest

from tests import engine_suite as es
from tests import traces_suite as ts


def test_off_changes_nothing(emu_engine):
    ts.off_changes_nothing(emu_engine)


def test_exact_against_numpy(emu_engine):
    ts.exact_against_numpy(emu_engine)


def test_batch_independence(emu_engine):
    ts.batch_independence(emu_engine, es.HostAsDevice())


def test_reset_rules(emu_engine):
    ts.reset_rules(emu_engine, es.HostAsDevice())


def test_peaks_random(emu_engine):
    ts.peaks_random(emu_engine, es.HostAsDevice())


def test_peaks_edges(emu_engine):
    ts.peaks_edges(emu_engine, es.HostAsDevice())


def test_two_tones_end_to_end(emu_engine):
    ts.two_tones_end_to_end(emu_engine, es.HostAsDevice())


@pytest.mark.gpu
def test_off_changes_nothing_gpu(gpu_engine):
    ts.off_changes_nothing(gpu_engine)


@pytest.mark.gpu
def test_exact_against_numpy_gpu(gpu_engine):
    ts.exact_against_numpy(gpu_engine)


@pytest.mark.gpu
def test_batch_independence_gpu(gpu_engine):
    ts.batch_independence(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_reset_rules_gpu(gpu_engine):
    ts.reset_rules(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_peaks_random_gpu(gpu_engine):
    ts.peaks_random(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_peaks_edges_gpu(gpu_engine):
    ts.peaks_edges(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_two_tones_end_to_end_gpu(gpu_engine):
    ts.two_tones_end_to_end(gpu_engine, es.TorchDevice())
