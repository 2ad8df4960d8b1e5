"""Frequency-mask trigger (DESIGN 3.10): each scenario of tests/mask_suite.py once on the CPU
emulation build of the engine sources and once, marked gpu, on the sm_100a library on the B200."""
import pytest

from tests import engine_suite as es
from tests import mask_suite as ms


def test_event_struct_layout():
    ms.abi_layout()


def test_off_changes_nothing(emu_engine):
    ms.off_changes_nothing(emu_engine)


def test_exact_against_oracle(emu_engine):
    ms.exact_against_oracle(emu_engine, es.HostAsDevice())


def test_mask_independent_of_batching(emu_engine):
    ms.batch_independence(emu_engine, es.HostAsDevice())


def test_capture(emu_engine):
    ms.capture(emu_engine, es.HostAsDevice())


def test_reset_and_error_rules(emu_engine):
    ms.reset_rules(emu_engine, es.HostAsDevice())


def test_burst_end_to_end(emu_engine):
    ms.burst_end_to_end(emu_engine)


@pytest.mark.gpu
def test_off_changes_nothing_gpu(gpu_engine):
    ms.off_changes_nothing(gpu_engine)


@pytest.mark.gpu
def test_exact_against_oracle_gpu(gpu_engine):
    ms.exact_against_oracle(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_mask_independent_of_batching_gpu(gpu_engine):
    ms.batch_independence(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_capture_gpu(gpu_engine):
    ms.capture(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_reset_and_error_rules_gpu(gpu_engine):
    ms.reset_rules(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_burst_end_to_end_gpu(gpu_engine):
    ms.burst_end_to_end(gpu_engine)
