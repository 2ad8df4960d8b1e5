"""Kernel + host logic of the engine on the CPU emulation build (tests/emu):
the SAME csrc sources nvcc compiles for sm_100a, run as fibers.  Proves the
indexing / hand-off / edge-case logic in the GPU-less container; numerical
parity proper is tests/test_gpu_parity.py on the B200."""
import pytest

from oracle import golden_cases as gc
from tests import engine_suite as es

EMU_CASES = [c["name"] for c in gc.CASES]


@pytest.mark.parametrize("name", EMU_CASES)
def test_golden_case(emu_engine, name):
    es.golden_case(emu_engine, name)


def test_ema_rows(emu_engine):
    es.ema_rows(emu_engine, 3)


def test_batch_equals_single(emu_engine, emu_lib):
    es.batch_equals_single(emu_engine, emu_lib)


def test_pipeline_equals_one_lane(emu_engine):
    es.pipeline_equals_one_lane(emu_engine, es.HostAsDevice())


def test_pipeline_equals_one_lane_other_wire_formats(emu_engine):
    # int16 IQ read by the FIR interior itself (each lane widens its own chunk ends), complex64
    from pypanadapter_b200 import synth
    es.pipeline_equals_one_lane(emu_engine, es.HostAsDevice(), nframes=9, w=synth.CFG2_CS16)
    es.pipeline_equals_one_lane(emu_engine, es.HostAsDevice(), nframes=9, w=synth.CFG1, n=2048 * 8 * 4 + 77)


def test_pipeline_channels_equal_plain(emu_engine):
    es.pipeline_channels_equal_plain(emu_engine, es.HostAsDevice())


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_pipeline_random_ops(emu_engine, seed):
    es.pipeline_random_ops(emu_engine, es.HostAsDevice(), seed=seed, nops=30)


def test_big_r16_parity(emu_engine):
    es.big_r16_parity(emu_engine, nframes=2)


def test_ema_batch_independent(emu_engine):
    es.ema_batch_independent(emu_engine)


def test_ring(emu_engine):
    es.ring_behaviour(emu_engine)


def test_decimated_chunk(emu_engine):
    es.decimated_chunk(emu_engine)


def test_plain_decimate_and_linear(emu_engine):
    es.plain_decimate_and_linear(emu_engine)


def test_error_paths(emu_engine):
    es.error_paths(emu_engine)


def test_f_demod(emu_engine):
    es.f_demod_extension(emu_engine)


def test_tile_geometries(emu_engine):
    es.tile_geometries(emu_engine)


# ---- buffer mirrors (Data / PSD / Waterfall) on the emulated engine ----------
from tests import buffers_suite as bs  # noqa: E402


def test_data_foldback(emu_engine):
    bs.data_foldback(emu_engine)


def test_data_random_sequences(emu_engine):
    bs.data_random_sequences(emu_engine, range(8))


def test_psd_update(emu_engine):
    bs.psd_update_matches_reference(emu_engine)


def test_psd_update_u8(emu_engine):
    bs.psd_update_u8(emu_engine)


def test_psd_update_cs16(emu_engine):
    bs.psd_update_cs16(emu_engine)


def test_rtl_tcp_source(emu_engine):
    bs.rtl_tcp_source(emu_engine)


def test_event_driven_run(emu_engine):
    bs.event_driven_run(emu_engine)


def test_psd_update_real(emu_engine):
    bs.psd_update_real(emu_engine)


def test_waterfall_image(emu_engine):
    bs.waterfall_image(emu_engine)


def test_waterfall_display(emu_engine):
    bs.waterfall_display(emu_engine)


def test_waterfall_random_shapes(emu_engine):
    bs.waterfall_random_shapes(emu_engine, range(4))


def test_level_mapping_edges(emu_engine):
    bs.level_mapping_edges(emu_engine)


def test_waterfall_engine_rows(emu_engine):
    bs.waterfall_from_engine_rows(emu_engine)


def test_scipy_shaped_calls(emu_engine):
    bs.scipy_shaped_calls(emu_engine)


# ---- ZFB_MODE_FAST ------------------------------------------------------------------
@pytest.mark.parametrize("name", es.FAST_CASES)
def test_fast_golden_case(emu_engine, name):
    es.fast_golden_case(emu_engine, name)


def test_fast_activation(emu_engine):
    es.fast_activation(emu_engine)


def test_fast_matches_exact_chunk(emu_engine):
    es.fast_matches_exact_chunk(emu_engine)


def test_fast_batch_and_ema(emu_engine):
    es.fast_batch_and_ema(emu_engine)


def test_fast_strong_out_of_band(emu_engine):
    es.fast_strong_out_of_band(emu_engine)


def test_fast_generic_fir_kernel(emu_engine):
    es.fast_generic_fir_kernel(emu_engine)


def test_cs16_wire_format(emu_engine):
    es.cs16_wire_format(emu_engine)


def test_multi_channel(emu_engine):
    es.multi_channel(emu_engine)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_configs(emu_engine, seed):
    es.random_configs(emu_engine, seed, 12)


def test_producer_consumer_threads(emu_engine):
    bs.producer_consumer_threads(emu_engine)


def test_reconfigure_stress(emu_engine):
    es.reconfigure_stress(emu_engine)


def test_replay_source(emu_engine):
    bs.replay_source_through_plugin_api(emu_engine)


def test_dropin_on_standin_modules(emu_engine):
    bs.dropin_on_standin_modules(emu_engine)


def test_fast_state_survives_frame_len(emu_engine):
    bs.fast_mode_state_survives_frame_len(emu_engine)


def test_ring_wrap_within_one_launch(emu_engine):
    bs.ring_wrap_within_one_launch(emu_engine)


def test_taper_design_and_preview(emu_engine):
    bs.taper_design_and_preview(emu_engine)
