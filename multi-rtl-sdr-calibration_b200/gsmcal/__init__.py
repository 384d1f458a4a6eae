"""gsmcal - B200-native GSM sync/calibration hot path of multi-rtl-sdr-calibration (host-side mirror).

The product is csrc/libgsmcal.so (hand-written sm_100a kernels behind the C ABI of include/gsmcal.h);
this package is the Python stand-in for the MATLAB call sites, used by the tests and bench.py.
"""
from .api import (BCCH_demod, FCCH_demod, SCH_demod, gsm_normal_training_sequence_gen,  # noqa: F401
                  FCCH_coarse_position, FCCH_fine_correction, GsmcalError, SCH_corr_rate_correction,  # noqa: F401
                  band_power, calibrate_batch, calibrate_batch_submit, calibrate_demod_batch, carrier_correct_post_SCH, chn_filter_4x, chn_filter_8x_4x,
                  chn_filter_taps, device_count, diversity_power_spectrum, fcch_scan, fir1, fir_filter, frame_clock_offsets,
                  gsm_SCH_training_sequence_gen,
                  launch_count, max_bursts, move_fft_snr_runtime_avg, move_fft_snr_trace, raw2iq, raw2iq_fir,
                  set_device, specific_fft_snr_fix_avg, total_ppm_calculation)
from . import ingest  # noqa: F401,E402  (rtl_tcp capture side: set_*_tcp, DongleIngest, calibrate_from_dongles)
