"""Channel power and occupied bandwidth (DESIGN 3.11): each scenario of tests/power_suite.py once on
the CPU emulation build of the engine sources and once, marked gpu, on the sm_100a library on the
B200."""
import pytest

from tests import engine_suite as es
from tests import power_suite as ps


def test_off_changes_nothing(emu_engine):
    ps.off_changes_nothing(emu_engine)


def test_exact_against_restatement(emu_engine):
    ps.exact_against_restatement(emu_engine, es.HostAsDevice())


def test_hz_bands_and_edges(emu_engine):
    ps.hz_mapping(emu_engine)


def test_parseval(emu_engine):
    ps.parseval(emu_engine)


def test_against_oracle_rows(emu_engine):
    ps.against_oracle_rows(emu_engine)


def test_power_independent_of_batching(emu_engine):
    ps.batch_independence(emu_engine, es.HostAsDevice())


def test_reset_and_error_rules(emu_engine):
    ps.reset_rules(emu_engine, es.HostAsDevice())


def test_burst_end_to_end(emu_engine):
    ps.burst_end_to_end(emu_engine)


@pytest.mark.gpu
def test_off_changes_nothing_gpu(gpu_engine):
    ps.off_changes_nothing(gpu_engine)


@pytest.mark.gpu
def test_exact_against_restatement_gpu(gpu_engine):
    ps.exact_against_restatement(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_hz_bands_and_edges_gpu(gpu_engine):
    ps.hz_mapping(gpu_engine)


@pytest.mark.gpu
def test_parseval_gpu(gpu_engine):
    ps.parseval(gpu_engine)


@pytest.mark.gpu
def test_against_oracle_rows_gpu(gpu_engine):
    ps.against_oracle_rows(gpu_engine)


@pytest.mark.gpu
def test_power_independent_of_batching_gpu(gpu_engine):
    ps.batch_independence(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_reset_and_error_rules_gpu(gpu_engine):
    ps.reset_rules(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_burst_end_to_end_gpu(gpu_engine):
    ps.burst_end_to_end(gpu_engine)
