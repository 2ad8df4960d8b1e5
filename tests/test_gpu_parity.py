"""Parity tests proper: the sm_100a library on a real B200, called through the
C ABI (ctypes), against the golden reference rows and the oracle.
Run with ``pytest -m gpu``.  Tolerances: tests/parity.py (0.01 dB20 above
-100 dBFS, argmax exact)."""
import numpy as np
import pytest

from oracle import golden_cases as gc
from oracle import zoompsd_oracle as zo
from pypanadapter_b200 import synth
from tests import engine_suite as es
from tests import parity

pytestmark = pytest.mark.gpu

ALL = [c["name"] for c in gc.CASES]


def test_product_library_is_sm100a(gpu_lib):
    assert gpu_lib.zfb_build_kind() == b"sm_100a"


@pytest.mark.parametrize("name", ALL)
def test_golden_case(gpu_engine, name):
    es.golden_case(gpu_engine, name)


def test_ema_rows(gpu_engine):
    es.ema_rows(gpu_engine, 4)


def test_ema_batch_independent(gpu_engine):
    es.ema_batch_independent(gpu_engine)


def test_slabs_equal_one_lane(gpu_engine):
    es.slabs_equal_one_lane(gpu_engine, es.TorchDevice())


def test_slabs_equal_one_lane_full_size(gpu_engine):
    """cfg2 at its full frame length, 160 frames in slabs of 40 across both lanes (several slabs per
    lane: the lanes' power sums are reused while the rows of earlier slabs are being finished)."""
    import torch
    w = synth.CFG2
    frames = synth.make_frames(w, 160, distinct=160)
    d_in = torch.from_numpy(frames).cuda()
    rows = {}
    for slabs in (1, 2):
        gpu_engine.set_option("slabs", slabs)
        gpu_engine.set_group(40)
        gpu_engine.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype="u8", flip=True,
                             crop="thread", ema_alpha=w.ema_alpha)
        gpu_engine.reset_ema()
        d_rows = torch.zeros((160, gpu_engine.row_width), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        for _ in range(3):                      # back-to-back batches: the EMA runs on across them
            gpu_engine.process_device(d_in.data_ptr(), 160, d_rows.data_ptr())
        gpu_engine.synchronize()
        assert gpu_engine.slab_lanes == slabs
        rows[slabs] = d_rows.cpu().numpy()
    gpu_engine.set_group(0)
    assert np.array_equal(rows[1], rows[2])
    assert np.isfinite(rows[2]).all()


def test_pipeline_equals_one_lane(gpu_engine):
    es.pipeline_equals_one_lane(gpu_engine, es.TorchDevice())


def test_pipeline_channels_equal_plain(gpu_engine):
    es.pipeline_channels_equal_plain(gpu_engine, es.TorchDevice())


@pytest.mark.parametrize("seed", range(6))
def test_pipeline_random_ops(gpu_engine, seed):
    es.pipeline_random_ops(gpu_engine, es.TorchDevice(), seed=seed, nops=60)


def test_pipeline_full_size_and_join_stream(gpu_engine):
    """cfg2 at full frame length: 12 pipelined batches of 48 frames back to back (both lanes busy,
    EMA carried on the finishing stream), a consumer on ANOTHER stream ordered by zfb_join(stream);
    rows equal the plain path's bit for bit."""
    import torch
    w = synth.CFG2
    nb, F = 12, 48
    frames = synth.make_frames(w, nb * F, distinct=nb * F)
    d_in = torch.from_numpy(frames).cuda()
    fbytes = frames[0].nbytes
    out = {}
    side = torch.cuda.Stream()
    for pipeline in (0, 1):
        gpu_engine.set_option("pipeline", pipeline)
        gpu_engine.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype="u8", flip=True,
                             crop="thread", ema_alpha=w.ema_alpha)
        gpu_engine.reset_ema()
        W = gpu_engine.row_width
        d_rows = torch.zeros((nb * F, W), dtype=torch.float32, device="cuda")
        copies = []
        torch.cuda.synchronize()
        for b in range(nb):
            gpu_engine.process_device(d_in.data_ptr() + b * F * fbytes, F, d_rows.data_ptr() + b * F * W * 4)
            if pipeline:
                gpu_engine.join(side.cuda_stream)            # only the side stream waits
                with torch.cuda.stream(side):
                    copies.append(d_rows[b * F:(b + 1) * F].clone())
        if pipeline:
            side.synchronize()
            assert gpu_engine.slab_lanes == 2
            got_side = torch.cat(copies, 0).cpu().numpy()
        gpu_engine.synchronize()
        out[pipeline] = d_rows.cpu().numpy()
    gpu_engine.set_option("pipeline", 0)
    assert np.array_equal(out[0], out[1])
    assert np.array_equal(got_side, out[0])
    assert np.isfinite(out[1]).all()


def test_big_cluster_equals_scratch(gpu_engine):
    es.big_cluster_equals_scratch(gpu_engine, nframes=5)


def test_batch_equals_single(gpu_engine, gpu_lib):
    es.batch_equals_single(gpu_engine, gpu_lib)


def test_ring(gpu_engine):
    es.ring_behaviour(gpu_engine)


def test_decimated_chunk(gpu_engine):
    es.decimated_chunk(gpu_engine)


def test_plain_decimate_and_linear(gpu_engine):
    es.plain_decimate_and_linear(gpu_engine)


def test_error_paths(gpu_engine):
    es.error_paths(gpu_engine)


def test_f_demod(gpu_engine):
    es.f_demod_extension(gpu_engine)


def test_cfg3_row_full_size(gpu_engine):
    """BASELINE configs[2]: one 2^20-sample row, 65536-pt Hann, 31 segments."""
    w = synth.CFG3
    x = synth.make_frame(w, 3)
    gpu_engine.configure(w.fs, w.fft_size, 1, len(x), w.window, crop=None)
    row = gpu_engine.process(x)[0].astype(np.float64)
    want = zo.zoom_psd(x, w.fs, w.fft_size, 1, w.window, crop=None)
    parity.assert_row_parity(row, want, parity.floor_db20(w.fs, w.window, w.fft_size, False), "cfg3")


@pytest.mark.parametrize("channel", [0, 37, 63])
def test_cfg4_channel_full_size(gpu_engine, channel):
    """BASELINE configs[3]: one of 64 virtual receivers over a 20 MS/s stream."""
    w = synth.CFG4
    x = synth.make_frame(w, 0)
    fc = float(synth.cfg4_centres()[channel])
    gpu_engine.configure(w.fs, w.fft_size, w.fft_ratio, len(x), w.window, f_demod=fc)
    row = gpu_engine.process(x)[0].astype(np.float64)
    want = zo.zoom_psd(x, w.fs, w.fft_size, w.fft_ratio, w.window, f_demod=fc)
    parity.assert_row_parity(row, want, parity.floor_db20(w.fs, w.window, w.fft_size, True),
                             "cfg4 ch%d" % channel)
    # the channel's own tone sits 7 kHz above its centre
    W = len(row)
    assert int(np.argmax(row)) == W // 2 + int(round(7000.0 / (w.fs / w.fft_ratio / w.fft_size)))


@pytest.mark.parametrize("N,R", [(1024, 64), (4096, 2), (16384, 4), (32768, 1), (131072, 1),
                                 (262144, 2)])
def test_sweep_corner(gpu_engine, N, R):
    """BASELINE configs[4] corners: decim 1..64 x N 1024..262144."""
    fs = 2.4e6
    # SURVEY 8d cfg5: avg = max(R, 16) -- down to ONE Welch segment at R = 64 (such rows take the
    # engine's fp64 path, zfb_precise.cuh; round 1 dodged them with >= 7 segments)
    avg = max(R, 16)
    n = N * avg
    x = gc.tone_noise(n, fs, [(0.013 * fs / R, 0.4), (-0.02 * fs / R, 0.03)], 2e-3, 900 + N % 97 + R,
                      np.complex64)
    gpu_engine.configure(fs, N, R, n, "hamming", crop="thread")
    row = gpu_engine.process(x)[0].astype(np.float64)
    want = zo.zoom_psd(x, fs, N, R, "hamming", crop="thread")
    parity.assert_row_parity(row, want, parity.floor_db20(fs, "hamming", N, R > 1), "N%d R%d" % (N, R))


@pytest.mark.parametrize("window", ["hann", "blackmanharris", "boxcar", ("kaiser", 8.6), "bartlett"])
def test_big_fft_detrend_with_dc(gpu_engine, window):
    """N = 65536 (radix-16 front pass): scipy.signal.welch's detrend='constant' (S:2111) is applied
    after the FFT there, X -= mean * FFT(window) -- through the few non-zero bins of a cosine-sum
    window or the dense table of any other -- so a chunk with a strong DC offset is the case to hold
    against the oracle."""
    fs, N = 2.4e6, 65536
    n = N * 5
    x = gc.tone_noise(n, fs, [(0.11 * fs, 0.3), (-0.23 * fs, 0.02)], 2e-3, 4242, np.complex64)
    x = (x + np.complex64(0.35 - 0.2j)).astype(np.complex64)
    gpu_engine.configure(fs, N, 1, n, window, crop=None)
    row = gpu_engine.process(x)[0].astype(np.float64)
    want = zo.zoom_psd(x, fs, N, 1, window, crop=None)
    parity.assert_row_parity(row, want, parity.floor_db20(fs, window, N, False), "N65536 dc %s" % (window,))


def test_device_path_equals_host_path(gpu_engine):
    """zfb_process_device on resident buffers == zfb_process_host, bit for bit,
    at a batch that spans several groups (size-independent property)."""
    import torch
    w = synth.CFG2
    frames = synth.make_frames(w, 40, distinct=4)
    gpu_engine.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype="u8",
                         flip=True, crop="thread")
    host_rows = gpu_engine.process(frames)
    d_in = torch.from_numpy(frames).cuda()
    d_rows = torch.empty((40, gpu_engine.row_width), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    gpu_engine.process_device(d_in.data_ptr(), 40, d_rows.data_ptr())
    gpu_engine.synchronize()
    dev_rows = d_rows.cpu().numpy()
    assert np.array_equal(dev_rows, host_rows)
    # repeated frames give identical rows (frames are independent)
    for i in range(4, 40):
        assert np.array_equal(host_rows[i], host_rows[i % 4])
    c = gpu_engine.counters()
    assert c["frames"] == 80 and c["kernels"] > 0


def test_tile_geometries(gpu_engine):
    es.tile_geometries(gpu_engine)


# ---- buffer mirrors (Data / PSD / Waterfall) on the GPU ------------------------
from tests import buffers_suite as bs  # noqa: E402


def test_data_foldback(gpu_engine):
    bs.data_foldback(gpu_engine)


def test_data_random_sequences(gpu_engine):
    bs.data_random_sequences(gpu_engine, range(8))


def test_psd_update(gpu_engine):
    bs.psd_update_matches_reference(gpu_engine)


def test_psd_update_u8(gpu_engine):
    bs.psd_update_u8(gpu_engine)


def test_psd_update_cs16(gpu_engine):
    bs.psd_update_cs16(gpu_engine)


def test_rtl_tcp_source(gpu_engine):
    bs.rtl_tcp_source(gpu_engine)


def test_event_driven_run(gpu_engine):
    bs.event_driven_run(gpu_engine)


def test_psd_update_real(gpu_engine):
    bs.psd_update_real(gpu_engine)


def test_waterfall_image(gpu_engine):
    bs.waterfall_image(gpu_engine)


def test_waterfall_display(gpu_engine):
    bs.waterfall_display(gpu_engine)


def test_waterfall_random_shapes(gpu_engine):
    bs.waterfall_random_shapes(gpu_engine, range(40))


def test_level_mapping_edges(gpu_engine):
    bs.level_mapping_edges(gpu_engine)


def test_waterfall_engine_rows(gpu_engine):
    bs.waterfall_from_engine_rows(gpu_engine)


def test_scipy_shaped_calls(gpu_engine):
    bs.scipy_shaped_calls(gpu_engine)


# ---- ZFB_MODE_FAST ------------------------------------------------------------------
@pytest.mark.parametrize("name", es.FAST_CASES)
def test_fast_golden_case(gpu_engine, name):
    es.fast_golden_case(gpu_engine, name)


def test_fast_activation(gpu_engine):
    es.fast_activation(gpu_engine)


def test_fast_matches_exact_chunk(gpu_engine):
    es.fast_matches_exact_chunk(gpu_engine)


def test_fast_batch_and_ema(gpu_engine):
    es.fast_batch_and_ema(gpu_engine)


def test_fast_strong_out_of_band(gpu_engine):
    es.fast_strong_out_of_band(gpu_engine)


def test_fast_generic_fir_kernel(gpu_engine):
    es.fast_generic_fir_kernel(gpu_engine)


def test_cs16_wire_format(gpu_engine):
    es.cs16_wire_format(gpu_engine)


def test_multi_channel(gpu_engine):
    es.multi_channel(gpu_engine)


@pytest.mark.parametrize("seed", [11, 12, 13, 14])
def test_random_configs(gpu_engine, seed):
    es.random_configs(gpu_engine, seed, 25)


def test_producer_consumer_threads(gpu_engine):
    bs.producer_consumer_threads(gpu_engine)


def test_reconfigure_stress(gpu_engine):
    es.reconfigure_stress(gpu_engine)


def test_replay_source(gpu_engine):
    bs.replay_source_through_plugin_api(gpu_engine)


def test_dropin_on_standin_modules(gpu_engine):
    bs.dropin_on_standin_modules(gpu_engine)


def test_fast_state_survives_frame_len(gpu_engine):
    bs.fast_mode_state_survives_frame_len(gpu_engine)


def test_ring_wrap_within_one_launch(gpu_engine):
    bs.ring_wrap_within_one_launch(gpu_engine)


def test_taper_design_and_preview(gpu_engine):
    bs.taper_design_and_preview(gpu_engine)
