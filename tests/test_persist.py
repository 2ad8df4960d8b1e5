"""Decaying persistence spectrum (DESIGN 3.9): each scenario of tests/persist_suite.py once on
the CPU emulation build of the engine sources and once, marked gpu, on the sm_100a library on
the B200."""
import pytest

from tests import engine_suite as es
from tests import persist_suite as ps


def test_off_changes_nothing(emu_engine):
    ps.off_changes_nothing(emu_engine)


def test_exact_against_oracle(emu_engine):
    ps.exact_against_oracle(emu_engine)


def test_persistence_independent_of_batching(emu_engine):
    ps.batch_independence(emu_engine, es.HostAsDevice())


def test_reset_rules(emu_engine):
    ps.reset_rules(emu_engine, es.HostAsDevice())


def test_persistence_image(emu_engine):
    ps.image(emu_engine, es.HostAsDevice())


def test_intermittent_tone_end_to_end(emu_engine):
    ps.intermittent_tone(emu_engine)


@pytest.mark.gpu
def test_off_changes_nothing_gpu(gpu_engine):
    ps.off_changes_nothing(gpu_engine)


@pytest.mark.gpu
def test_exact_against_oracle_gpu(gpu_engine):
    ps.exact_against_oracle(gpu_engine)


@pytest.mark.gpu
def test_persistence_independent_of_batching_gpu(gpu_engine):
    ps.batch_independence(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_reset_rules_gpu(gpu_engine):
    ps.reset_rules(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_persistence_image_gpu(gpu_engine):
    ps.image(gpu_engine, es.TorchDevice())


@pytest.mark.gpu
def test_intermittent_tone_end_to_end_gpu(gpu_engine):
    ps.intermittent_tone(gpu_engine)
