"""ctypes binding of libhabdec_b200.so (include/habdec_b200.h) plus a thin Python mirror of the
reference Decoder interface (code/Decoder/Decoder.h:65-141) used by tests and bench.

The library is CUDA only: importing works anywhere (so the CPU test tier can check the exported
symbols), creating a decoder without a B200-class device raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HBD_LIB") or os.path.join(_HERE, "libhabdec_b200.so")   # HBD_LIB: tuning variants

HBD_OK, HBD_ERR_ARG, HBD_ERR_CUDA, HBD_ERR_STATE, HBD_ERR_NOMEM = 0, -1, -2, -3, -4
STAGE_DECIMATED, STAGE_FILTERED, STAGE_DEMOD, STAGE_LPTAPS, STAGE_PENDING, STAGE_BITS = 0, 1, 2, 5, 6, 7

# input sample formats (hbd_iq_format): interleaved I, Q, little endian
IQ_CF32, IQ_CS16, IQ_CS8, IQ_CU8 = 0, 1, 2, 3
IQ_BYTES = {IQ_CF32: 8, IQ_CS16: 4, IQ_CS8: 2, IQ_CU8: 2}          # per complex sample
_IQ_DTYPE = {IQ_CF32: np.float32, IQ_CS16: np.int16, IQ_CS8: np.int8, IQ_CU8: np.uint8}


def dequantise(q, fmt: int) -> np.ndarray:
    """The value the decoder sees for integer IQ `q` ([..., 2] or [..., 2n] interleaved I, Q of the format's dtype):
    CS16 v / 32768, CS8 v / 128, CU8 (v - 128) / 128; complex64 [...]/[..., n].  Every value is exact in float32."""
    q = np.asarray(q)
    if fmt == IQ_CF32:
        return np.ascontiguousarray(q, dtype=np.float32).view(np.complex64).reshape(q.shape[:-1] + (-1,))
    if q.dtype != _IQ_DTYPE[fmt]:
        raise ValueError("format %d needs %s samples, got %s" % (fmt, np.dtype(_IQ_DTYPE[fmt]).name, q.dtype))
    v = q.astype(np.float64)
    v = v / 32768.0 if fmt == IQ_CS16 else (v / 128.0 if fmt == IQ_CS8 else (v - 128.0) / 128.0)
    return np.ascontiguousarray(v.astype(np.float32)).view(np.complex64).reshape(q.shape[:-1] + (-1,))


def quantise(iq, fmt: int, scale: float = 1.0):
    """Integer IQ of the format from complex samples: round(iq * scale * 2^k) (+ 128 for CU8), clipped to the format's range;
    interleaved [..., 2n].  numpy in -> numpy out, torch in -> torch out (on the tensor's device)."""
    if fmt == IQ_CF32:
        raise ValueError("quantise makes integer formats")
    full = {IQ_CS16: 32768.0, IQ_CS8: 128.0, IQ_CU8: 128.0}[fmt]
    lo, hi = (-32768, 32767) if fmt == IQ_CS16 else ((-128, 127) if fmt == IQ_CS8 else (0, 255))
    off = 128.0 if fmt == IQ_CU8 else 0.0
    if not isinstance(iq, np.ndarray) and type(iq).__module__.startswith("torch"):
        import torch
        ri = torch.view_as_real(iq.to(torch.complex64)).reshape(*iq.shape[:-1], -1)
        dt = {IQ_CS16: torch.int16, IQ_CS8: torch.int8, IQ_CU8: torch.uint8}[fmt]
        return torch.clamp(torch.round(ri * float(scale * full)) + off, lo, hi).to(dt)
    iq = np.asarray(iq, dtype=np.complex64)
    ri = iq.view(np.float32).reshape(iq.shape[:-1] + (-1,)).astype(np.float64)
    return np.clip(np.round(ri * (scale * full)) + off, lo, hi).astype(_IQ_DTYPE[fmt])


class SpectrumInfo(C.Structure):
    _fields_ = [("min_", C.c_float), ("max_", C.c_float), ("noise_floor_", C.c_double), ("noise_variance_", C.c_double),
                ("sampling_rate_", C.c_double), ("shift_", C.c_double), ("peak_left_", C.c_int), ("peak_right_", C.c_int),
                ("peak_left_valid_", C.c_int), ("peak_right_valid_", C.c_int)]


class SsdvPacketInfo(C.Structure):
    _fields_ = [("callsign", C.c_char * 8), ("image_id", C.c_int), ("packet_id", C.c_int), ("width", C.c_int),
                ("height", C.c_int), ("errors", C.c_int), ("set_size", C.c_int)]


class Telemetry(C.Structure):
    _fields_ = [("payload_callsign", C.c_char * 64), ("datetime", C.c_char * 40), ("frame", C.c_int), ("lat", C.c_float),
                ("lon", C.c_float), ("alt", C.c_float)]


class GpsDistance(C.Structure):
    _fields_ = [("dist_line_", C.c_double), ("dist_circle_", C.c_double), ("dist_radians_", C.c_double),
                ("elevation_", C.c_double), ("bearing_", C.c_double)]


class ChannelStats(C.Structure):
    _fields_ = [("num_ok_", C.c_uint), ("D_", GpsDistance), ("dist_max_", C.c_double), ("elev_min_", C.c_double), ("age_s", C.c_double)]


class ResultRecord(C.Structure):
    """hbd_result_record: the 256-byte wire format of the multi-GPU result gather (include/habdec_b200.h)."""
    _fields_ = [("channel", C.c_uint32), ("n_chars", C.c_uint16), ("sentence_bytes", C.c_uint16), ("n_sentences", C.c_uint16),
                ("flags", C.c_uint16), ("peak_left", C.c_int32), ("peak_right", C.c_int32), ("frequency_correction", C.c_float),
                ("shift", C.c_float), ("noise_floor", C.c_float), ("noise_variance", C.c_float), ("reserved", C.c_uint32),
                ("chars", C.c_char * 88), ("sentences", C.c_char * 128)]


RECORD_BYTES = C.sizeof(ResultRecord)


class ScanParams(C.Structure):
    _fields_ = [("min_snr_db", C.c_double), ("min_shift_hz", C.c_double), ("max_shift_hz", C.c_double), ("max_tone_ratio_db", C.c_double)]


class BaudEstimate(C.Structure):
    _fields_ = [("baud", C.c_double), ("nominal", C.c_double), ("confidence", C.c_double), ("runs", C.c_uint), ("long_runs", C.c_uint)]


# hbd_baud_estimate as a numpy record (BatchDecoder.baud_estimates)
BAUD_ESTIMATE_DTYPE = np.dtype([("baud", np.float64), ("nominal", np.float64), ("confidence", np.float64), ("runs", np.uint32),
                                ("long_runs", np.uint32)])
assert BAUD_ESTIMATE_DTYPE.itemsize == C.sizeof(BaudEstimate)


class ScanSignal(C.Structure):
    _fields_ = [("center_hz", C.c_double), ("shift_hz", C.c_double), ("snr_db", C.c_double), ("bin_lo", C.c_int), ("bin_hi", C.c_int)]

TELEMETRY_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(Telemetry), C.c_char_p)
SSDV_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(SsdvPacketInfo), C.POINTER(C.c_ubyte))
SENTENCE_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p)
CHARS_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_char), C.c_size_t)

# name -> (restype, argtypes); this table is also what the CPU test tier checks against the header
_H = C.c_void_p
SIGNATURES = {
    "hbd_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(_H)]),
    "hbd_destroy": (None, [_H]),
    "hbd_last_error": (C.c_char_p, [_H]),
    "hbd_set_stream": (C.c_int, [_H, C.c_void_p]),
    "hbd_set_record": (C.c_int, [_H, C.c_int]),
    "hbd_set_fft_size": (C.c_int, [_H, C.c_size_t]),
    "hbd_set_baud": (C.c_int, [_H, C.c_int, C.c_double]),
    "hbd_get_baud": (C.c_double, [_H, C.c_int]),
    "hbd_set_rtty_bits": (C.c_int, [_H, C.c_int, C.c_size_t]),
    "hbd_get_rtty_bits": (C.c_size_t, [_H, C.c_int]),
    "hbd_set_rtty_stops": (C.c_int, [_H, C.c_int, C.c_float]),
    "hbd_get_rtty_stops": (C.c_float, [_H, C.c_int]),
    "hbd_set_lowpass_bw": (C.c_int, [_H, C.c_int, C.c_float]),
    "hbd_get_lowpass_bw": (C.c_float, [_H, C.c_int]),
    "hbd_set_lowpass_trans": (C.c_int, [_H, C.c_int, C.c_float]),
    "hbd_get_lowpass_trans": (C.c_float, [_H, C.c_int]),
    "hbd_set_dc_remove": (C.c_int, [_H, C.c_int, C.c_int]),
    "hbd_get_dc_remove": (C.c_int, [_H, C.c_int]),
    "hbd_setup_decimation_factor": (C.c_size_t, [_H, C.c_size_t]),
    "hbd_setup_decimation_bw": (C.c_size_t, [_H, C.c_double]),
    "hbd_push_samples": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_size_t, C.c_double]),
    "hbd_push_samples_batch": (C.c_int, [_H, C.c_void_p, C.c_size_t, C.c_size_t, C.c_double]),
    "hbd_push_samples_device": (C.c_int, [_H, C.c_void_p, C.c_size_t, C.c_size_t, C.c_double]),
    "hbd_set_nco": (C.c_int, [_H, C.c_int, C.c_double]),
    "hbd_get_nco": (C.c_double, [_H, C.c_int]),
    "hbd_afc_retune": (C.c_int, [_H, C.c_double, C.c_void_p]),
    "hbd_push_wideband": (C.c_int, [_H, C.c_void_p, C.c_size_t, C.c_double]),
    "hbd_push_wideband_device": (C.c_int, [_H, C.c_void_p, C.c_size_t, C.c_double]),
    "hbd_push_iq": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_int, C.c_size_t, C.c_double]),
    "hbd_push_iq_batch": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, C.c_double]),
    "hbd_push_iq_device": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, C.c_double]),
    "hbd_push_iq_wideband": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_size_t, C.c_double]),
    "hbd_push_iq_wideband_device": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_size_t, C.c_double]),
    "hbd_process": (C.c_int, [_H]),
    "hbd_process_async": (C.c_int, [_H]),
    "hbd_collect": (C.c_int, [_H]),
    "hbd_collect_ready": (C.c_int, [_H, C.c_uint]),
    "hbd_synchronize": (C.c_int, [_H]),
    "hbd_reset_channels": (C.c_int, [_H, C.c_void_p, C.c_size_t]),
    "hbd_kernel_launches": (C.c_ulonglong, [_H]),
    "hbd_set_kernel_timing": (C.c_int, [_H, C.c_int]),
    "hbd_get_kernel_timing": (C.c_int, [_H, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_uint)]),
    "hbd_get_rtty": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_get_last_sentence": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_poll_chars": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_poll_sentences": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_poll_raw_chars": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_set_raw_chars": (C.c_int, [_H, C.c_int]),
    "hbd_set_host_threads": (C.c_int, [_H, C.c_int]),
    "hbd_set_sentence_callback": (C.c_int, [_H, SENTENCE_CB, C.c_void_p]),
    "hbd_set_chars_callback": (C.c_int, [_H, CHARS_CB, C.c_void_p]),
    "hbd_set_ssdv": (C.c_int, [_H, C.c_int]),
    "hbd_set_ssdv_callback": (C.c_int, [_H, SSDV_CB, C.c_void_p]),
    "hbd_poll_ssdv_packets": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t]),
    "hbd_get_ssdv_image": (C.c_size_t, [_H, C.c_int, C.c_char_p, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_get_ssdv_last_image": (C.c_int, [_H, C.c_int, C.c_char_p, C.POINTER(C.c_int)]),
    "hbd_ssdv_check_packets": (C.c_int, [_H, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "hbd_ssdv_host_replay": (C.c_size_t, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "hbd_get_decimation_factor": (C.c_int, [_H]),
    "hbd_get_input_sampling_rate": (C.c_double, [_H]),
    "hbd_get_decimated_sampling_rate": (C.c_double, [_H]),
    "hbd_get_symbol_rate": (C.c_double, [_H, C.c_int]),
    "hbd_n_channels": (C.c_int, [_H]),
    "hbd_get_bins_count": (C.c_size_t, [_H]),
    "hbd_get_fft": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_get_demodulated": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_get_power_spectrum": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_get_peaks": (C.c_int, [_H, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "hbd_get_noise_floor": (C.c_int, [_H, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "hbd_get_shift": (C.c_double, [_H, C.c_int]),
    "hbd_get_frequency_correction": (C.c_double, [_H, C.c_int]),
    "hbd_reset_frequency_correction": (C.c_int, [_H, C.c_int, C.c_double]),
    "hbd_get_spectrum_info": (C.c_size_t, [_H, C.c_int, C.POINTER(SpectrumInfo), C.c_void_p, C.c_size_t]),
    "hbd_get_stats_batch": (C.c_size_t, [_H, C.c_void_p, C.c_size_t]),
    "hbd_get_spectrum_frame": (C.c_size_t, [_H, C.c_int, C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_get_spectrum_frames": (C.c_size_t, [_H, C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "hbd_set_demod_accumulate": (C.c_int, [_H, C.c_int]),
    "hbd_get_demod_frame": (C.c_size_t, [_H, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_get_demod_frames": (C.c_size_t, [_H, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "hbd_record_set": (None, [C.c_void_p, C.c_uint32, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "hbd_pack_results": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_set_stats_snapshot": (C.c_int, [_H, C.c_int]),
    "hbd_sink_create": (C.c_void_p, [C.c_int]),
    "hbd_sink_destroy": (None, [C.c_void_p]),
    "hbd_sink_feed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "hbd_sink_set_threads": (C.c_int, [C.c_void_p, C.c_int]),
    "hbd_sink_poll_chars": (C.c_size_t, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_sink_poll_sentences": (C.c_size_t, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_sink_stats": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "hbd_sink_totals": (None, [C.c_void_p] + [C.POINTER(C.c_ulonglong)] * 4),
    "hbd_sink_hash": (C.c_uint64, [C.c_void_p]),
    "hbd_dist_unique_id": (C.c_int, [C.c_void_p]),
    "hbd_dist_init": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p]),
    "hbd_dist_use_comm": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_int]),
    "hbd_dist_finalize": (C.c_int, [_H]),
    "hbd_dist_total_channels": (C.c_int, [_H]),
    "hbd_gather_results": (C.c_int, [_H, C.c_void_p]),
    "hbd_parse_sentence": (C.c_int, [C.c_char_p, C.c_longlong, C.POINTER(Telemetry)]),
    "hbd_parse_sentence_time": (C.c_int, [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_float)]),
    "hbd_parse_gps_pos": (C.c_int, [C.c_char_p, C.POINTER(C.c_float)]),
    "hbd_timestamp_from_hms": (C.c_size_t, [C.c_int, C.c_int, C.c_float, C.c_longlong, C.c_char_p, C.c_size_t]),
    "hbd_calc_gps_distance": (None, [C.c_double] * 6 + [C.POINTER(GpsDistance)]),
    "hbd_tracking_telemetry_payload": (C.c_size_t, [C.POINTER(Telemetry), C.c_char_p, C.c_size_t]),
    "hbd_tracker_create": (C.c_void_p, []),
    "hbd_tracker_destroy": (None, [C.c_void_p]),
    "hbd_tracker_set_station": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_float]),
    "hbd_tracker_set_clock": (C.c_int, [C.c_void_p, C.c_longlong]),
    "hbd_tracker_set_callback": (C.c_int, [C.c_void_p, TELEMETRY_CB, C.c_void_p]),
    "hbd_tracker_push": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p]),
    "hbd_tracker_push_sentence": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p]),
    "hbd_tracker_poll": (C.c_size_t, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_tracker_reset": (C.c_int, [C.c_void_p, C.c_int]),
    "hbd_tracker_stats": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ChannelStats)]),
    "hbd_tracker_stats_payload": (C.c_size_t, [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_size_t]),
    "hbd_tracker_get_sentence": (C.c_size_t, [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_size_t]),
    "hbd_attach_tracker": (C.c_int, [_H, C.c_void_p, C.c_int]),
    "hbd_scanner_create": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(C.c_void_p)]),
    "hbd_scanner_destroy": (None, [C.c_void_p]),
    "hbd_scanner_last_error": (C.c_char_p, [C.c_void_p]),
    "hbd_scanner_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hbd_scan_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_double]),
    "hbd_scan_push_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_double]),
    "hbd_scan_reset": (C.c_int, [C.c_void_p]),
    "hbd_scan_get_psd": (C.c_size_t, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_ulonglong)]),
    "hbd_scan_default_params": (None, [C.POINTER(ScanParams)]),
    "hbd_scan_find": (C.c_int, [C.c_void_p, C.POINTER(ScanParams), C.c_void_p, C.c_size_t]),
    "hbd_scan_detect": (C.c_int, [C.c_void_p, C.c_size_t, C.c_double, C.POINTER(ScanParams), C.c_void_p, C.c_size_t]),
    "hbd_set_baud_estimation": (C.c_int, [_H, C.c_int]),
    "hbd_get_baud_estimates": (C.c_int, [_H, C.c_void_p, C.c_size_t]),
    "hbd_apply_baud_estimates": (C.c_int, [_H, C.c_double, C.c_uint, C.c_void_p]),
    "hbd_get_baud_histogram": (C.c_size_t, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_debug_stage": (C.c_size_t, [_H, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "hbd_design_lowpass": (C.c_size_t, [C.c_float, C.c_float, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t]),
    "hbd_extract_sentence": (C.c_int, [C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "hbd_crc16": (None, [C.c_char_p, C.c_size_t, C.c_char_p]),
    "hbd_text_replay": (C.c_size_t, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
}

_lib = None


def load():
    """Load the shared library (raises if it was not built: there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(habdec_b200 has no CPU or pure-Python compute path)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            if os.environ.get("HBD_LIB") and not hasattr(lib, name):
                continue              # an older tuning / comparison build (tools/ab_step.py)
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class HbdError(RuntimeError):
    pass


def design_lowpass(rel_width: float, trans: float, input_size: int, current_taps: int = 0) -> np.ndarray:
    lib = load()
    out = np.zeros(4096, dtype=np.float32)
    n = lib.hbd_design_lowpass(rel_width, trans, input_size, current_taps, out.ctypes.data, out.size)
    return out[:n] if n != current_taps else out[:0]


def extract_sentence(stream: bytes):
    lib = load()
    cs, data, crc = (C.create_string_buffer(len(stream) + 8) for _ in range(3))
    rest = C.c_size_t(0)
    ok = lib.hbd_extract_sentence(stream, len(stream), cs, data, crc, len(stream) + 8, C.byref(rest))
    if not ok:
        return None
    return cs.value, data.value, crc.value, rest.value


def ssdv_host_replay(chunks: list[bytes], accepted: list[tuple]):
    """Host half of the SSDV path alone: chunks = the per-call raw characters, accepted = [(pos, packet256, errors)]
    ascending.  Returns [(chunk index, callsign, image_id, packet_id, width, height, errors, set_size, packet)]."""
    lib = load()
    chars = b"".join(chunks)
    sizes = (C.c_size_t * max(len(chunks), 1))(*[len(c) for c in chunks])
    cbuf = (C.c_ubyte * max(len(chars), 1)).from_buffer_copy(chars or b"\0")
    na = len(accepted)
    pos = (C.c_uint * max(na, 1))(*[a[0] & 0xFFFFFFFF for a in accepted])
    pk = (C.c_ubyte * max(256 * na, 1)).from_buffer_copy(b"".join(a[1] for a in accepted) or b"\0")
    er = (C.c_int * max(na, 1))(*[a[2] for a in accepted])
    cap = len(chars) // 256 + 1
    infos = (SsdvPacketInfo * cap)()
    which = (C.c_uint * cap)()
    out = (C.c_ubyte * (256 * cap))()
    n = lib.hbd_ssdv_host_replay(cbuf, sizes, len(chunks), pos, pk, er, na, infos, which, out, cap)
    raw = bytes(out)
    return [(which[k], infos[k].callsign.decode(), infos[k].image_id, infos[k].packet_id, infos[k].width, infos[k].height,
             infos[k].errors, infos[k].set_size, raw[256 * k:256 * k + 256]) for k in range(n)]


def text_replay(chunks: list[bytes]):
    """The text layer alone (host only): (CRC-valid sentences, last sentence, remaining text stream) after feeding `chunks`."""
    lib = load()
    chars = b"".join(chunks)
    sizes = (C.c_size_t * max(len(chunks), 1))(*[len(c) for c in chunks])
    cbuf = (C.c_ubyte * max(len(chars), 1)).from_buffer_copy(chars or b"\0")
    n = lib.hbd_text_replay(cbuf, sizes, len(chunks), None, 0)
    out = C.create_string_buffer(max(n, 1))
    lib.hbd_text_replay(cbuf, sizes, len(chunks), out, n)
    sent, last, stream = out.raw[:n].split(b"\x1e")
    return [x for x in sent.split(b"\n") if x], last, stream


def crc16(s: bytes) -> bytes:
    lib = load()
    out = C.create_string_buffer(5)
    lib.hbd_crc16(s, len(s), out)
    return out.value


# ---- telemetry layer (host only; code/common/sentence_parse.cpp, GpsDistance.cpp, websocketServer/main.cpp:292-366) ----
def parse_sentence(sentence: bytes, now_unix: int = -1):
    """(status, dict | None): status 1 = parsed, 0 = rejected (empty optional), -1 = the reference throws here."""
    t = Telemetry()
    rc = load().hbd_parse_sentence(sentence, int(now_unix), C.byref(t))
    return rc, (_telemetry_dict(t) if rc == 1 else None)


def _telemetry_dict(t: Telemetry) -> dict:
    return {"payload_callsign": t.payload_callsign, "datetime": t.datetime, "frame": t.frame, "lat": t.lat, "lon": t.lon, "alt": t.alt,
            "tracking": tracking_payload(t)}


def tracking_payload(t: Telemetry) -> bytes:
    buf = C.create_string_buffer(256)
    load().hbd_tracking_telemetry_payload(C.byref(t), buf, 256)
    return buf.value


def parse_sentence_time(s: bytes):
    h, m, sec = C.c_int(), C.c_int(), C.c_float()
    rc = load().hbd_parse_sentence_time(s, C.byref(h), C.byref(m), C.byref(sec))
    return rc, ((h.value, m.value, sec.value) if rc == 1 else None)


def parse_gps_pos(s: bytes):
    v = C.c_float()
    rc = load().hbd_parse_gps_pos(s, C.byref(v))
    return rc, (v.value if rc == 1 else None)


def timestamp_from_hms(h: int, m: int, s: float, now_unix: int = -1) -> bytes:
    buf = C.create_string_buffer(96)
    load().hbd_timestamp_from_hms(int(h), int(m), float(s), int(now_unix), buf, 96)
    return buf.value


def calc_gps_distance(lat1, lon1, alt1, lat2, lon2, alt2) -> GpsDistance:
    g = GpsDistance()
    load().hbd_calc_gps_distance(lat1, lon1, alt1, lat2, lon2, alt2, C.byref(g))
    return g


def make_records(channel0: int, chars: list[bytes], sentences: list[bytes], stats=None) -> np.ndarray:
    """Host-only packer (hbd_record_set): one record per channel from the HEADS of its character / sentence streams.
    Returns (records uint8[n, 256], chars_used[n], sentence_bytes_used[n])."""
    lib = load()
    n = len(chars)
    recs = np.zeros((n, RECORD_BYTES), dtype=np.uint8)
    cu, su = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
    for i in range(n):
        a, b = C.c_size_t(0), C.c_size_t(0)
        st = np.asarray(stats[i] if stats is not None else np.zeros(6), dtype=np.float64)
        lib.hbd_record_set(recs[i].ctypes.data, channel0 + i, chars[i], len(chars[i]), sentences[i], len(sentences[i]), st.ctypes.data, C.byref(a), C.byref(b))
        cu[i], su[i] = a.value, b.value
    return recs, cu, su


class ResultSink:
    """Rank-0 side of the result gather (hbd_result_sink, host only): fed with records, polled like a decoder."""

    def __init__(self, total_channels: int):
        self._lib = load()
        self._s = C.c_void_p(self._lib.hbd_sink_create(int(total_channels)))
        self.total_channels = total_channels

    def close(self):
        if self._s:
            self._lib.hbd_sink_destroy(self._s)
            self._s = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self): return self._s

    def feed(self, records: np.ndarray) -> int:
        r = np.ascontiguousarray(records, dtype=np.uint8).reshape(-1, RECORD_BYTES)
        return self._lib.hbd_sink_feed(self._s, r.ctypes.data, r.shape[0])

    def _take(self, fn, ch):
        n = fn(self._s, ch, None, 0)
        if not n:
            return b""
        buf = C.create_string_buffer(n)
        fn(self._s, ch, buf, n)
        return buf.raw[:n]

    def poll_chars(self, ch: int) -> bytes: return self._take(self._lib.hbd_sink_poll_chars, ch)
    def poll_sentences(self, ch: int) -> list[bytes]:
        return [x for x in self._take(self._lib.hbd_sink_poll_sentences, ch).split(b"\n") if x]

    def stats(self, ch: int):
        out = np.zeros(6, dtype=np.float64)
        return out if self._lib.hbd_sink_stats(self._s, ch, out.ctypes.data) == HBD_OK else None

    def totals(self) -> dict:
        v = [C.c_ulonglong(0) for _ in range(4)]
        self._lib.hbd_sink_totals(self._s, *[C.byref(x) for x in v])
        return {"chars": v[0].value, "sentences": v[1].value, "sentences_min": v[2].value, "records": v[3].value}

    def hash(self) -> int: return int(self._lib.hbd_sink_hash(self._s))


def dist_unique_id() -> bytes:
    """128 bytes that rank 0 hands to every other rank before hbd_dist_init (ncclGetUniqueId)."""
    buf = (C.c_ubyte * 128)()
    rc = load().hbd_dist_unique_id(buf)
    if rc != HBD_OK:
        raise HbdError("hbd_dist_unique_id failed (%d): NCCL could not be loaded" % rc)
    return bytes(buf)


class Tracker:
    """SentenceCallback + GLOBALS::STATS for many channels (hbd_tracker); host only."""

    def __init__(self, station=None, now_unix: int = -1):
        self._lib = load()
        self._t = C.c_void_p(self._lib.hbd_tracker_create())
        self._cb = None
        if station is not None:
            self.set_station(*station)
        if now_unix >= 0:
            self.set_clock(now_unix)

    def close(self):
        if self._t:
            self._lib.hbd_tracker_destroy(self._t)
            self._t = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self): return self._t
    def set_station(self, lat, lon, alt): self._lib.hbd_tracker_set_station(self._t, float(lat), float(lon), float(alt))
    def set_clock(self, now_unix: int): self._lib.hbd_tracker_set_clock(self._t, int(now_unix))
    def push(self, ch: int, callsign: bytes, data: bytes, crc: bytes) -> int: return self._lib.hbd_tracker_push(self._t, ch, callsign, data, crc)
    def push_sentence(self, ch: int, sentence: bytes) -> int: return self._lib.hbd_tracker_push_sentence(self._t, ch, sentence)
    def reset(self, ch: int):
        """Forget channel `ch`: its stats, sentences map and unpolled records (hbd_tracker_reset)."""
        if self._lib.hbd_tracker_reset(self._t, int(ch)) != HBD_OK:
            raise HbdError("hbd_tracker_reset failed")

    def set_callback(self, fn):
        self._cb = TELEMETRY_CB(lambda user, ch, t, s: fn(ch, _telemetry_dict(t.contents), s)) if fn else C.cast(None, TELEMETRY_CB)
        self._lib.hbd_tracker_set_callback(self._t, self._cb, None)

    def poll(self, ch: int) -> list[dict]:
        n = self._lib.hbd_tracker_poll(self._t, ch, None, 0)
        if not n:
            return []
        arr = (Telemetry * n)()
        self._lib.hbd_tracker_poll(self._t, ch, arr, n)
        return [_telemetry_dict(t) for t in arr]

    def stats(self, ch: int) -> ChannelStats:
        st = ChannelStats()
        self._lib.hbd_tracker_stats(self._t, ch, C.byref(st))
        return st

    def stats_payload(self, ch: int, with_age: bool = False) -> bytes:
        buf = C.create_string_buffer(512)
        self._lib.hbd_tracker_stats_payload(self._t, ch, int(with_age), buf, 512)
        return buf.value

    def get_sentence(self, ch: int, frame: int) -> bytes:
        buf = C.create_string_buffer(1200)
        n = self._lib.hbd_tracker_get_sentence(self._t, ch, int(frame), buf, 1200)
        return buf.value if n else b""


# ---- wideband scanner (hbd_scanner / hbd_scan_*): where the RTTY payloads of a capture are -------------------------
def scan_default_params() -> dict:
    p = ScanParams()
    load().hbd_scan_default_params(C.byref(p))
    return {name: getattr(p, name) for name, _ in ScanParams._fields_}


def _scan_params(params: dict):
    if not params:
        return None
    p = ScanParams(**scan_default_params())
    for k, v in params.items():
        if k not in scan_default_params():
            raise TypeError("unknown scan parameter %r" % k)
        setattr(p, k, float(v))
    return C.byref(p)


def _scan_signals(call) -> list[dict]:
    arr = (ScanSignal * 16)()
    n = call(arr, len(arr))
    if n > len(arr):                  # more than the first guess: once more with room for all
        arr = (ScanSignal * n)()
        n = call(arr, n)
    if n < 0:
        raise HbdError("scan detection failed (%d)" % n)
    return [{"center_hz": x.center_hz, "shift_hz": x.shift_hz, "snr_db": x.snr_db, "bin_lo": x.bin_lo, "bin_hi": x.bin_hi} for x in arr[:n]]


def scan_detect(psd, fs: float, **params) -> list[dict]:
    """Tone pairs in an fft-shifted float32 PSD (hbd_scan_detect, host only); params as hbd_scan_params (defaults when absent)."""
    psd = np.ascontiguousarray(psd, dtype=np.float32)
    lib, p = load(), _scan_params(params)
    return _scan_signals(lambda out, cap: lib.hbd_scan_detect(psd.ctypes.data, psd.size, float(fs), p, out, cap))


class Scanner:
    """Averaged GPU spectrum of a wideband capture and the RTTY tone pairs in it (hbd_scanner).  Offsets are relative to the
    capture centre, in the units BatchDecoder.set_nco takes."""

    def __init__(self, n_fft: int, device: int = 0):
        self._lib = load()
        h = C.c_void_p()
        rc = self._lib.hbd_scanner_create(int(device), int(n_fft), C.byref(h))
        if rc != HBD_OK:
            raise HbdError("hbd_scanner_create failed (%d): n_fft must be a power of two in [4096, 2^20], and a CUDA device "
                           "(B200, sm_100a) is required" % rc)
        self._s = h
        self.n_fft = int(n_fft)
        self.fs = None

    def close(self):
        if getattr(self, "_s", None):
            self._lib.hbd_scanner_destroy(self._s)
            self._s = None

    __del__ = close

    def _chk(self, rc):
        if rc != HBD_OK:
            raise HbdError("habdec_b200 scanner error %d: %s" % (rc, (self._lib.hbd_scanner_last_error(self._s) or b"").decode()))

    def set_stream(self, cuda_stream_ptr: int): self._chk(self._lib.hbd_scanner_set_stream(self._s, cuda_stream_ptr))

    def push(self, iq, fs: float, fmt: int = IQ_CF32):
        """iq: complex64 [n] (IQ_CF32) or interleaved integers [2n] of the format's dtype"""
        if fmt == IQ_CF32:
            arr = np.ascontiguousarray(iq, dtype=np.complex64)
            n = arr.size
        else:
            arr = BatchDecoder._iq_arr(iq, fmt, 1)
            n = arr.size // 2
        self._chk(self._lib.hbd_scan_push(self._s, arr.ctypes.data, int(fmt), n, float(fs)))
        self.fs = float(fs)

    def push_device(self, ptr: int, n: int, fs: float, fmt: int = IQ_CF32):
        self._chk(self._lib.hbd_scan_push_device(self._s, ptr, int(fmt), int(n), float(fs)))
        self.fs = float(fs)

    def reset(self):
        self._chk(self._lib.hbd_scan_reset(self._s))
        self.fs = None

    def psd(self):
        """(float32 [n_fft] fft-shifted PSD, segments averaged)"""
        out = np.empty(self.n_fft, dtype=np.float32)
        seg = C.c_ulonglong(0)
        if self._lib.hbd_scan_get_psd(self._s, out.ctypes.data, out.size, C.byref(seg)) != self.n_fft:
            raise HbdError("hbd_scan_get_psd failed: %s" % (self._lib.hbd_scanner_last_error(self._s) or b"").decode())
        return out, seg.value

    def freqs(self) -> np.ndarray:
        """Offset of every PSD bin from the capture centre in Hz (needs the sampling rate of a push)."""
        if self.fs is None:
            raise HbdError("no sampling rate latched yet: push first")
        return (np.arange(self.n_fft, dtype=np.float64) - self.n_fft // 2) * (self.fs / self.n_fft)

    def find(self, **params) -> list[dict]:
        """[{center_hz, shift_hz, snr_db, bin_lo, bin_hi}] sorted by center_hz"""
        p = _scan_params(params)
        return _scan_signals(lambda out, cap: self._lib.hbd_scan_find(self._s, p, out, cap))


class BatchDecoder:
    """N independent channels on one GPU; method names follow habdec::Decoder (Decoder.h:65-141)."""

    def __init__(self, n_channels: int, device: int = 0, baud: float = 300.0, rtty_bits: int = 8, rtty_stops: float = 2.0,
                 lowpass_bw: float = 1500.0, lowpass_trans: float = 0.025, dec_factor: int = 256, dc_remove: bool = False,
                 record: bool = False, fft_bins: int = 4096):
        self._lib = load()
        h = _H()
        rc = self._lib.hbd_create(n_channels, device, C.byref(h))
        if rc != HBD_OK:
            raise HbdError(f"hbd_create failed ({rc}): a CUDA device (B200, sm_100a) is required, there is no CPU fallback")
        self._h = h
        self.n_channels = n_channels
        self._cbs = []
        # same order as code/websocketServer/main.cpp:544-553
        self.baud(baud); self.rtty_bits(rtty_bits); self.rtty_stops(rtty_stops); self.dc_remove(dc_remove)
        self.lowpass_bw(lowpass_bw); self.lowpass_trans(lowpass_trans)
        if record:
            self._chk(self._lib.hbd_set_record(self._h, 1))
        if fft_bins != 4096:
            self.set_fft_size(fft_bins)
        if self.setupDecimationStagesFactor(dec_factor) != dec_factor:
            raise HbdError("unsupported decimation factor %r" % dec_factor)

    # ---- plumbing
    def _chk(self, rc):
        if rc != HBD_OK:
            raise HbdError("habdec_b200 error %d: %s" % (rc, (self._lib.hbd_last_error(self._h) or b"").decode()))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.hbd_destroy(self._h)
            self._h = None

    __del__ = close

    def set_fft_size(self, n_bins: int): self._chk(self._lib.hbd_set_fft_size(self._h, int(n_bins)))

    def set_stream(self, cuda_stream_ptr: int):
        self._chk(self._lib.hbd_set_stream(self._h, cuda_stream_ptr))

    # ---- configuration
    def baud(self, v, ch=-1): self._chk(self._lib.hbd_set_baud(self._h, ch, float(v)))
    def rtty_bits(self, v, ch=-1): self._chk(self._lib.hbd_set_rtty_bits(self._h, ch, int(v)))
    def rtty_stops(self, v, ch=-1): self._chk(self._lib.hbd_set_rtty_stops(self._h, ch, float(v)))
    def lowpass_bw(self, v, ch=-1): self._chk(self._lib.hbd_set_lowpass_bw(self._h, ch, float(v)))
    def lowpass_trans(self, v, ch=-1): self._chk(self._lib.hbd_set_lowpass_trans(self._h, ch, float(v)))
    def dc_remove(self, v, ch=-1): self._chk(self._lib.hbd_set_dc_remove(self._h, ch, int(bool(v))))
    def setupDecimationStagesFactor(self, factor: int) -> int: return self._lib.hbd_setup_decimation_factor(self._h, int(factor))
    def setupDecimationStagesBW(self, max_rate: float) -> int: return self._lib.hbd_setup_decimation_bw(self._h, float(max_rate))
    def getDecimationFactor(self): return self._lib.hbd_get_decimation_factor(self._h)
    def getInputSamplingRate(self): return self._lib.hbd_get_input_sampling_rate(self._h)
    def getDecimatedSamplingRate(self): return self._lib.hbd_get_decimated_sampling_rate(self._h)

    # ---- feed
    def pushSamples(self, ch: int, iq: np.ndarray, fs: float):
        iq = np.ascontiguousarray(iq, dtype=np.complex64)
        self._chk(self._lib.hbd_push_samples(self._h, ch, iq.ctypes.data, iq.size, float(fs)))

    def pushSamplesBatch(self, iq: np.ndarray, fs: float):
        """iq: complex64 [n_channels, n]"""
        assert iq.ndim == 2 and iq.shape[0] == self.n_channels and iq.dtype == np.complex64
        pitch = iq.strides[0] // 8
        assert iq.strides[1] == 8
        self._chk(self._lib.hbd_push_samples_batch(self._h, iq.ctypes.data, iq.shape[1], pitch, float(fs)))

    def pushSamplesDevice(self, ptr: int, n: int, pitch: int, fs: float):
        self._chk(self._lib.hbd_push_samples_device(self._h, ptr, n, pitch, float(fs)))

    # ---- NCO pre-mixer / wideband channeliser (include/habdec_b200.h)
    def set_nco(self, freq_hz: float, ch=-1): self._chk(self._lib.hbd_set_nco(self._h, ch, float(freq_hz)))
    def get_nco(self, ch=0) -> float: return self._lib.hbd_get_nco(self._h, ch)

    def afc_retune(self, min_abs_hz: float = 100.0) -> np.ndarray:
        """Close the AFC loop for all channels on the GPU; returns the applied corrections [n_channels] (0 = none)."""
        out = np.zeros(self.n_channels, dtype=np.float64)
        rc = self._lib.hbd_afc_retune(self._h, float(min_abs_hz), out.ctypes.data)
        if rc < 0:
            self._chk(rc)
        return out

    # ---- baud-rate estimation (hbd_set_baud_estimation ..., the estimator is stated in include/habdec_b200.h)
    def set_baud_estimation(self, on): self._chk(self._lib.hbd_set_baud_estimation(self._h, int(bool(on))))

    def baud_estimates(self) -> np.ndarray:
        """Every channel's estimate as of all calls so far: a BAUD_ESTIMATE_DTYPE array [n_channels]."""
        out = np.zeros(self.n_channels, dtype=BAUD_ESTIMATE_DTYPE)
        rc = self._lib.hbd_get_baud_estimates(self._h, out.ctypes.data, out.size)
        if rc < 0:
            self._chk(rc)
        return out

    def apply_baud_estimates(self, min_confidence: float = 0.8, min_runs: int = 100) -> np.ndarray:
        """Set each confident channel's baud to its nominal rate; returns the rates set [n_channels] (0 = unchanged)."""
        out = np.zeros(self.n_channels, dtype=np.float64)
        rc = self._lib.hbd_apply_baud_estimates(self._h, float(min_confidence), int(min_runs), out.ctypes.data)
        if rc < 0:
            self._chk(rc)
        return out

    def baud_histogram(self, ch: int) -> np.ndarray:
        """The channel's run histogram H[0 .. Lmax] (test hook; empty while estimation is off or before the first push)."""
        n = self._lib.hbd_get_baud_histogram(self._h, int(ch), None, 0)
        out = np.zeros(n, dtype=np.uint32)
        if n and self._lib.hbd_get_baud_histogram(self._h, int(ch), out.ctypes.data, n) != n:
            raise HbdError("hbd_get_baud_histogram failed: %s" % (self._lib.hbd_last_error(self._h) or b"").decode())
        return out

    def pushWideband(self, iq: np.ndarray, fs: float):
        """iq: complex64 [n], pushed to every channel through its NCO"""
        iq = np.ascontiguousarray(iq, dtype=np.complex64)
        self._chk(self._lib.hbd_push_wideband(self._h, iq.ctypes.data, iq.size, float(fs)))

    def pushWidebandDevice(self, ptr: int, n: int, fs: float):
        self._chk(self._lib.hbd_push_wideband_device(self._h, ptr, n, float(fs)))

    # ---- integer IQ input (hbd_push_iq*): arrays are interleaved I, Q of the format's dtype, [..., 2n]
    @staticmethod
    def _iq_arr(arr, fmt, ndim):
        arr = np.ascontiguousarray(arr, dtype=_IQ_DTYPE[fmt])
        assert arr.ndim == ndim and arr.shape[-1] % 2 == 0, "interleaved I, Q expected"
        return arr

    def pushIQ(self, ch: int, arr: np.ndarray, fmt: int, fs: float):
        arr = self._iq_arr(arr, fmt, 1)
        self._chk(self._lib.hbd_push_iq(self._h, ch, arr.ctypes.data, int(fmt), arr.shape[-1] // 2, float(fs)))

    def pushIQBatch(self, arr: np.ndarray, fmt: int, fs: float):
        """arr: [n_channels, n, 2] or [n_channels, 2n] (rows may be a strided view of a wider matrix)"""
        arr = np.asarray(arr)
        if arr.ndim == 3:
            arr = arr.reshape(arr.shape[0], -1)
        assert arr.ndim == 2 and arr.shape[0] == self.n_channels and arr.dtype == _IQ_DTYPE[fmt]
        assert arr.strides[1] == arr.itemsize and arr.strides[0] % IQ_BYTES[fmt] == 0
        self._chk(self._lib.hbd_push_iq_batch(self._h, arr.ctypes.data, int(fmt), arr.shape[1] // 2, arr.strides[0] // IQ_BYTES[fmt], float(fs)))

    def pushIQDevice(self, ptr: int, fmt: int, n: int, pitch: int, fs: float):
        self._chk(self._lib.hbd_push_iq_device(self._h, ptr, int(fmt), n, pitch, float(fs)))

    def pushIQWideband(self, arr: np.ndarray, fmt: int, fs: float):
        arr = self._iq_arr(arr, fmt, 1)
        self._chk(self._lib.hbd_push_iq_wideband(self._h, arr.ctypes.data, int(fmt), arr.shape[-1] // 2, float(fs)))

    def pushIQWidebandDevice(self, ptr: int, fmt: int, n: int, fs: float):
        self._chk(self._lib.hbd_push_iq_wideband_device(self._h, ptr, int(fmt), n, float(fs)))

    # ---- run
    def process(self): self._chk(self._lib.hbd_process(self._h))
    __call__ = process
    def process_async(self): self._chk(self._lib.hbd_process_async(self._h))
    def collect(self): self._chk(self._lib.hbd_collect(self._h))
    def collect_ready(self, lag: int): self._chk(self._lib.hbd_collect_ready(self._h, int(lag)))
    def synchronize(self): self._chk(self._lib.hbd_synchronize(self._h))

    def reset_channels(self, chs):
        """Channels `chs` start over like a new decoder with the same settings (hbd_reset_channels): calls in flight are
        drained first, unpolled output stays queued, the configuration and NCO frequency are kept."""
        arr = np.ascontiguousarray(np.atleast_1d(np.asarray(chs, dtype=np.int32)))
        self._chk(self._lib.hbd_reset_channels(self._h, arr.ctypes.data, arr.size))
    def kernel_launches(self) -> int: return int(self._lib.hbd_kernel_launches(self._h))
    def set_kernel_timing(self, on): self._chk(self._lib.hbd_set_kernel_timing(self._h, int(on)))   # 0 off, 1 K1 only, 2 K1 + rest of step
    def kernel_timing(self, which: int):
        """(total_ms, count) since set_kernel_timing: K1 (which=0) or the rest of the step (which=1) with their launches; 5: the
        drains' host replay and calls drained; 6: host planning of the calls and frame counters stepped (hbd_get_kernel_timing)."""
        ms, cnt = C.c_double(0), C.c_uint(0)
        self._chk(self._lib.hbd_get_kernel_timing(self._h, which, C.byref(ms), C.byref(cnt)))
        return ms.value, cnt.value

    # ---- results
    def _bytes(self, fn, ch) -> bytes:
        n = fn(self._h, ch, None, 0)
        if not n:
            return b""
        buf = C.create_string_buffer(n)
        fn(self._h, ch, buf, n)
        return buf.raw[:n]

    def getRTTY(self, ch=0) -> bytes: return self._bytes(self._lib.hbd_get_rtty, ch)
    def getLastSentence(self, ch=0) -> bytes: return self._bytes(self._lib.hbd_get_last_sentence, ch)
    def poll_chars(self, ch=0) -> bytes: return self._bytes(self._lib.hbd_poll_chars, ch)
    def poll_raw_chars(self, ch=0) -> bytes: return self._bytes(self._lib.hbd_poll_raw_chars, ch)
    def set_host_threads(self, n: int): self._chk(self._lib.hbd_set_host_threads(self._h, int(n)))
    def set_raw_chars(self, on: bool): self._chk(self._lib.hbd_set_raw_chars(self._h, int(on)))
    def poll_sentences(self, ch=0) -> list[bytes]:
        return [s for s in self._bytes(self._lib.hbd_poll_sentences, ch).split(b"\n") if s]

    def attach_tracker(self, tracker, ch_offset: int = 0):
        self._tracker = tracker   # keep it alive
        self._chk(self._lib.hbd_attach_tracker(self._h, tracker.handle if tracker else None, int(ch_offset)))

    def set_sentence_callback(self, fn):
        cb = SENTENCE_CB(lambda user, ch, cs, data, crc: fn(ch, cs, data, crc))
        self._cbs.append(cb)
        self._chk(self._lib.hbd_set_sentence_callback(self._h, cb, None))

    # ---- SSDV packet sync (SSDV_wraper_t::push, ssdv_wrapper.cpp:37-148) ----
    def set_ssdv(self, on: bool = True): self._chk(self._lib.hbd_set_ssdv(self._h, int(on)))

    def set_ssdv_callback(self, fn):
        """fn(ch, info_dict, packet_bytes) per accepted packet, like ssdv_callback_ (Decoder.h:631-632)."""
        def tramp(_user, ch, info, pkt):
            i = info.contents
            fn(ch, dict(callsign=i.callsign.decode(), image_id=i.image_id, packet_id=i.packet_id, width=i.width, height=i.height,
                        errors=i.errors, set_size=i.set_size), bytes(pkt[:256]))
        self._ssdv_cb = SSDV_CB(tramp) if fn else SSDV_CB()
        self._chk(self._lib.hbd_set_ssdv_callback(self._h, self._ssdv_cb, None))

    def poll_ssdv_packets(self, ch=0) -> list[tuple]:
        """[(callsign, image_id, packet_id, width, height, errors, set_size, packet bytes)] since the previous poll."""
        n = self._lib.hbd_poll_ssdv_packets(self._h, ch, None, None, 0)
        if not n:
            return []
        infos = (SsdvPacketInfo * n)()
        pk = (C.c_ubyte * (256 * n))()
        self._lib.hbd_poll_ssdv_packets(self._h, ch, infos, pk, n)
        raw = bytes(pk)
        return [(i.callsign.decode(), i.image_id, i.packet_id, i.width, i.height, i.errors, i.set_size, raw[256 * k:256 * k + 256])
                for k, i in enumerate(infos)]

    def get_ssdv_image(self, ch: int, callsign: str, image_id: int) -> bytes:
        n = self._lib.hbd_get_ssdv_image(self._h, ch, callsign.encode(), int(image_id), None, 0)
        buf = (C.c_ubyte * max(n, 1))()
        self._lib.hbd_get_ssdv_image(self._h, ch, callsign.encode(), int(image_id), buf, n)
        return bytes(buf[:n])

    def get_ssdv_last_image(self, ch=0):
        cs = C.create_string_buffer(8)
        iid = C.c_int(0)
        self._chk(self._lib.hbd_get_ssdv_last_image(self._h, ch, cs, C.byref(iid)))
        return cs.value.decode(), iid.value

    def ssdv_check_packets(self, windows: np.ndarray):
        """Batch packet test on the GPU: windows uint8[n, 256] -> (verdict int32[n], errors int32[n], corrected uint8[n, 256])."""
        w = np.ascontiguousarray(windows, dtype=np.uint8).reshape(-1, 256).copy()
        n = w.shape[0]
        verdict = np.zeros(n, dtype=np.int32)
        errors = np.zeros(n, dtype=np.int32)
        self._chk(self._lib.hbd_ssdv_check_packets(self._h, w.ctypes.data, n, verdict.ctypes.data, errors.ctypes.data))
        return verdict, errors, w

    def set_chars_callback(self, fn):
        cb = CHARS_CB(lambda user, ch, p, n: fn(ch, C.string_at(p, n)))
        self._cbs.append(cb)
        self._chk(self._lib.hbd_set_chars_callback(self._h, cb, None))

    # ---- GUI data
    def _floats(self, fn, ch, *extra, complex_=False) -> np.ndarray:
        n = fn(self._h, ch, *extra, None, 0)
        out = np.empty(n, dtype=np.float32)
        if n:
            fn(self._h, ch, *extra, out.ctypes.data, n)
        return out.view(np.complex64) if complex_ else out

    def getBinsCount(self): return self._lib.hbd_get_bins_count(self._h)
    def getFFT(self, ch=0): return self._floats(self._lib.hbd_get_fft, ch, complex_=True)
    def getDemodulated(self, ch=0): return self._floats(self._lib.hbd_get_demodulated, ch)
    def getPowerSpectrum(self, ch=0): return self._floats(self._lib.hbd_get_power_spectrum, ch)
    def getPeaks(self, ch=0):
        pl, pr = C.c_int(0), C.c_int(0)
        self._chk(self._lib.hbd_get_peaks(self._h, ch, C.byref(pl), C.byref(pr)))
        return pl.value, pr.value
    def getNoiseFloor(self, ch=0):
        nf, nv = C.c_double(0), C.c_double(0)
        self._chk(self._lib.hbd_get_noise_floor(self._h, ch, C.byref(nf), C.byref(nv)))
        return nf.value, nv.value
    def getShift(self, ch=0): return self._lib.hbd_get_shift(self._h, ch)
    def getFrequencyCorrection(self, ch=0): return self._lib.hbd_get_frequency_correction(self._h, ch)
    def resetFrequencyCorrection(self, corr, ch=0): self._chk(self._lib.hbd_reset_frequency_correction(self._h, ch, float(corr)))
    def getSpectrumInfo(self, ch=0):
        info = SpectrumInfo()
        power = np.empty(self.getBinsCount(), dtype=np.float32)
        n = self._lib.hbd_get_spectrum_info(self._h, ch, C.byref(info), power.ctypes.data, power.size)
        return info, power[:n]

    # ---- websocket wire formats (PWR_ / DEM_ payloads, habdec_ws_protocol.cpp:353-429)
    def spectrum_frame(self, ch: int, zoom: float, resolution: int, type_size: int) -> bytes:
        n = self._lib.hbd_get_spectrum_frame(self._h, ch, zoom, resolution, type_size, None, 0)
        buf = C.create_string_buffer(max(n, 1))
        self._lib.hbd_get_spectrum_frame(self._h, ch, zoom, resolution, type_size, buf, n)
        return buf.raw[:n]

    def _frames(self, fn, *args) -> list[bytes]:
        sizes = np.zeros(self.n_channels, dtype=np.uint32)
        longest = fn(self._h, *args, None, 0, sizes.ctypes.data)
        if not longest:
            return [b""] * self.n_channels
        out = np.zeros((self.n_channels, longest), dtype=np.uint8)
        fn(self._h, *args, out.ctypes.data, longest, sizes.ctypes.data)
        return [out[c, :sizes[c]].tobytes() for c in range(self.n_channels)]

    def spectrum_frames(self, zoom: float, resolution: int, type_size: int) -> list[bytes]:
        return self._frames(self._lib.hbd_get_spectrum_frames, zoom, resolution, type_size)

    def set_demod_accumulate(self, on: bool): self._chk(self._lib.hbd_set_demod_accumulate(self._h, int(on)))

    def demod_frame(self, ch: int, resolution: int, type_size: int) -> bytes:
        n = self._lib.hbd_get_demod_frame(self._h, ch, resolution, type_size, None, 0)
        buf = C.create_string_buffer(max(n, 1))
        self._lib.hbd_get_demod_frame(self._h, ch, resolution, type_size, buf, n)
        return buf.raw[:n]

    def demod_frames(self, resolution: int, type_size: int) -> list[bytes]:
        return self._frames(self._lib.hbd_get_demod_frames, resolution, type_size)

    # ---- multi-GPU result gather (SURVEY 8e)
    def pack_results(self, ch_offset: int = 0) -> np.ndarray:
        """uint8[n_channels, 256]: one hbd_result_record per channel; consumes the pending characters / sentences."""
        recs = np.zeros((self.n_channels, RECORD_BYTES), dtype=np.uint8)
        n = self._lib.hbd_pack_results(self._h, int(ch_offset), recs.ctypes.data, self.n_channels)
        if n != self.n_channels:
            raise HbdError("hbd_pack_results failed: %s" % (self._lib.hbd_last_error(self._h) or b"").decode())
        return recs

    def set_stats_snapshot(self, on: bool = True): self._chk(self._lib.hbd_set_stats_snapshot(self._h, int(on)))

    def dist_init(self, rank: int, world: int, unique_id: bytes | None):
        buf = (C.c_ubyte * 128).from_buffer_copy(unique_id) if unique_id else None
        self._chk(self._lib.hbd_dist_init(self._h, int(rank), int(world), buf))

    def dist_finalize(self): self._chk(self._lib.hbd_dist_finalize(self._h))
    def dist_total_channels(self) -> int: return self._lib.hbd_dist_total_channels(self._h)

    def gather_results(self, sink: "ResultSink | None") -> int:
        if sink is not None:
            self._sinks = getattr(self, "_sinks", [])
            if sink not in self._sinks:
                self._sinks.append(sink)      # the sink borrows the handle's receive buffers: it has to outlive the handle
        rc = self._lib.hbd_gather_results(self._h, sink.handle if sink is not None else None)
        if rc < 0:
            self._chk(rc)
        return rc

    def stats_all(self) -> np.ndarray:
        """[n_channels, 6] float64: frequency correction, shift, noise floor, noise variance, peak left, peak right."""
        out = np.zeros((self.n_channels, 6), dtype=np.float64)
        self._lib.hbd_get_stats_batch(self._h, out.ctypes.data, out.size)
        return out

    def debug_stage(self, ch, stage) -> np.ndarray:
        return self._floats(self._lib.hbd_debug_stage, ch, stage, complex_=stage in (STAGE_DECIMATED, STAGE_FILTERED))
