"""ctypes mirror of include/soundgen_b200.h (struct layouts and prototypes)."""
from __future__ import annotations

import ctypes as C
import os

i32, i64, f64, f32 = C.c_int32, C.c_int64, C.c_double, C.c_float

SGB_OK = 0
SGB_ERR_INVALID, SGB_ERR_CUDA, SGB_ERR_UNSUPPORTED = -1, -2, -3
SGB_ERR_SYNTH, SGB_ERR_STREAM, SGB_ERR_STATE = -4, -5, -6
SGB_CONTOUR_LOESS, SGB_CONTOUR_SPLINE = 0, 1
SGB_OUT_F32, SGB_OUT_PCM16 = 0, 1
SGB_WIN_HAMMING, SGB_WIN_HANNING = 0, 1
SGB_CMP_COR, SGB_CMP_COSINE, SGB_CMP_DTW = 0, 1, 2
SGB_CMP_DTW_MAX_FRAMES = 4096

SYL_DOUBLES = ['attackLen', 'nonlinBalance', 'jitterDep', 'jitterLen', 'vibratoFreq',
               'vibratoDep', 'shimmerDep', 'rolloff', 'rolloffOct', 'rolloffKHz', 'rolloffParab',
               'rolloffParabHarm', 'rolloff_perAmpl', 'temperature', 'pitchDriftDep',
               'pitchDriftFreq', 'randomWalk_trendStrength', 'shortestEpoch', 'subFreq', 'subDep',
               'samplingRate', 'pitchFloor', 'pitchCeiling', 'pitchSamplingRate', 'throwaway']


class Syllable(C.Structure):
    _fields_ = [('kind', i32), ('silent_len', i32), ('pitch_off', i64), ('pitch_len', i32),
                ('pause_after', i32), ('z_off', i64), ('z_cap', i32), ('ampl_n', i32),
                ('ampl_off', i64), ('ampl_method', i32), ('pitch_anchor_n', i32),
                ('pitch_anchor_off', i64), ('pitch_method', i32), ('reserved0', i32),
                ('pitch_scale', f64)] + [(n, f64) for n in SYL_DOUBLES]


class Envelope(C.Structure):
    _fields_ = [('n_formants', i32), ('tracks_given', i32), ('formant_off', i64),
                ('mouth_n', i32), ('nc_fixed', i32), ('mouth_off', i64),
                ('mouth_method', i32), ('reserved0', i32), ('formantDep', f64), ('rolloffLip', f64), ('mouthOpenThres', f64),
                ('openMouthBoost', f64), ('vocalTract', f64), ('samplingRate', f64),
                ('speedSound', f64), ('smoothLinearFactor', f64)]


class Noise(C.Structure):
    _fields_ = [('len', i32), ('insertion', i32), ('mix', i32), ('wl', i32), ('u_off', i64),
                ('anchor_off', i64), ('anchor_n', i32), ('env_id', i32),
                ('strength_pre_off', i64), ('anchor_method', i32), ('reserved0', i32),
                ('rolloffNoise', f64), ('attackLen', f64),
                ('samplingRate', f64), ('overlap', f64)]


class Bout(C.Structure):
    _fields_ = [('syl_begin', i32), ('syl_end', i32), ('noise_begin', i32), ('noise_end', i32),
                ('env_id', i32), ('moving', i32), ('wl', i32), ('lead_silence', i32),
                ('tail_silence', i32), ('aglobal_n', i32), ('aglobal_off', i64),
                ('aglobal_method', i32), ('reserved0', i32), ('overlap', f64), ('amDep', f64), ('amFreq', f64), ('amShape', f64),
                ('samplingRate', f64), ('throwaway', f64)]


class Call(C.Structure):
    _fields_ = [('bout_begin', i32), ('bout_end', i32)]


class FormantRef(C.Structure):
    _fields_ = [('off', i64), ('n', i32), ('pad', i32)]


class BatchDesc(C.Structure):
    _fields_ = [('n_calls', i32), ('n_bouts', i32), ('n_syllables', i32), ('n_noises', i32),
                ('n_envelopes', i32), ('n_formant_refs', i32),
                ('calls', C.c_void_p), ('bouts', C.c_void_p), ('syllables', C.c_void_p),
                ('noises', C.c_void_p), ('envelopes', C.c_void_p), ('formant_index', C.c_void_p),
                ('pitch', C.c_void_p), ('n_pitch', i64),
                ('anchors', C.c_void_p), ('n_anchors', i64),
                ('formants', C.c_void_p), ('n_formants', i64),
                ('z', C.c_void_p), ('n_z', i64),
                ('u', C.c_void_p), ('n_u', i64),
                ('u_is_float', i32), ('reserved', i32),
                ('pre', C.c_void_p), ('n_pre', i64)]


class AnchorArg(C.Structure):
    _fields_ = [('time', C.c_void_p), ('value', C.c_void_p), ('n', i32), ('reserved', i32)]


class FormantArg(C.Structure):
    _fields_ = [('time', C.c_void_p), ('freq', C.c_void_p), ('amp', C.c_void_p), ('width', C.c_void_p),
                ('n_time', i32), ('n_freq', i32), ('n_amp', i32), ('n_width', i32)]


SG_DOUBLES = ['repeatBout', 'nSyl', 'sylLen', 'pauseLen', 'temperature', 'maleFemale', 'creakyBreathy',
              'nonlinBalance', 'nonlinDep', 'jitterLen', 'jitterDep', 'vibratoFreq', 'vibratoDep', 'shimmerDep',
              'attackLen', 'rolloff', 'rolloffOct', 'rolloffKHz', 'rolloffParab', 'rolloffParabHarm', 'rolloffLip',
              'formantDep', 'formantDepStoch', 'vocalTract', 'subFreq', 'subDep', 'shortestEpoch', 'amDep',
              'amFreq', 'amShape', 'rolloffNoise', 'samplingRate', 'windowLength', 'overlap', 'addSilence',
              'pitchFloor', 'pitchCeiling', 'pitchSamplingRate', 'throwaway']
SG_ANCHORS = ['pitchAnchors', 'pitchAnchorsGlobal', 'noiseAnchors', 'mouthAnchors', 'amplAnchors',
              'amplAnchorsGlobal']
TEMP_EFFECTS = ['sylLenDep', 'formDrift', 'formDisp', 'pitchDriftDep', 'pitchDriftFreq', 'pitchAnchorsDep',
                'noiseAnchorsDep', 'amplAnchorsDep']


class SoundgenArgs(C.Structure):
    _fields_ = [(n, f64) for n in SG_DOUBLES] + [('tempEffects', f64 * 8)] + \
               [(n, AnchorArg) for n in SG_ANCHORS] + \
               [('formants', C.c_void_p), ('n_formants', i32), ('reserved0', i32),
                ('formantsNoise', C.c_void_p), ('n_formantsNoise', i32), ('invalidArgAction', i32),
                ('contour_method', i32), ('rng_mode', i32), ('seed', C.c_uint32), ('sample_rejection', i32),
                ('rng_state', C.c_void_p),
                ('z', C.c_void_p), ('z_len', C.c_void_p), ('n_z', i32), ('device_pitch', i32),
                ('u', C.c_void_p), ('u_len', C.c_void_p), ('n_u', i32), ('reserved1', i32)]


class DeviceOut(C.Structure):
    _fields_ = [('dst', C.c_void_p), ('dst_elems', i64), ('dst_off', C.c_void_p), ('cap', C.c_void_p),
                ('out_written', C.c_void_p), ('stream', C.c_void_p), ('format', i32), ('reserved', i32)]


class SpecParams(C.Structure):
    _fields_ = [('wl', i32), ('window', i32), ('overlap', f64), ('n_bands', i32), ('db', i32), ('db_floor', f64),
                ('band_lo', C.c_void_p), ('band_len', C.c_void_p), ('band_w', C.c_void_p)]


class CompareParams(C.Structure):
    _fields_ = [('method', i32), ('n_feat', i32), ('pad', f64)]


T_NAMES = ['h2d', 'control', 'ampl', 'synth', 'compose', 'noise', 'assemble', 'envelope',
           'filter', 'finalize', 'd2h', 'total']


class RunInfo(C.Structure):
    _fields_ = [('total_samples', i64), ('synth_partials', i64), ('synth_samples', i64),
                ('filter_samples', i64), ('filter_frames', i64), ('noise_samples', i64),
                ('kernel_launches', i32), ('n_failed', i32), ('ms', f32 * len(T_NAMES))]


class SylArtefacts(C.Structure):
    _fields_ = [('nGC', i32), ('nHarmonics', i32), ('rows_kept', i32), ('nEpochs', i32),
                ('n_upsampled', i32), ('n_jitter_idx', i32), ('z_used', i32), ('status', i32),
                ('raw_max', f64)]


EXPORTS = ['sgb_version', 'sgb_last_error', 'sgb_device_count', 'sgb_set_device', 'sgb_pin', 'sgb_unpin', 'sgb_device_pci_bus_id',
           'sgb_measure_fp32_peak',
           'sgb_batch_create', 'sgb_batch_destroy', 'sgb_batch_upload', 'sgb_batch_run',
           'sgb_batch_lengths', 'sgb_batch_fetch_f32', 'sgb_batch_fetch_f64', 'sgb_batch_fetch_pcm16', 'sgb_batch_status',
           'sgb_batch_export', 'sgb_rows_export', 'sgb_spec_frames', 'sgb_batch_spectrogram', 'sgb_rows_spectrogram',
           'sgb_rows_compare', 'sgb_param_range',
           'sgb_batch_syllable_len', 'sgb_batch_syllable_fetch', 'sgb_batch_noise_fetch',
           'sgb_batch_artefacts', 'sgb_batch_artefact_ints', 'sgb_batch_pitch_per_gc', 'sgb_batch_checksums', 'sgb_batch_debug_state',
           'sgb_get_rolloff', 'sgb_get_spectral_envelope', 'sgb_filter_len', 'sgb_filter',
           'sgb_batch_run_begin', 'sgb_batch_run_finish', 'sgb_batch_bout_geometry', 'sgb_batch_set_tracks',
           'sgb_batch_z_used', 'sgb_abi_sizes', 'sgb_synth_min_rows_set', 'sgb_host_set_threads', 'sgb_frontend_create', 'sgb_frontend_destroy', 'sgb_frontend_add', 'sgb_frontend_add_seeded', 'sgb_frontend_add_many', 'sgb_frontend_clear',
           'sgb_frontend_round_begin', 'sgb_frontend_resolve', 'sgb_frontend_round_end', 'sgb_frontend_round_calls',
           'sgb_frontend_status', 'sgb_frontend_warnings', 'sgb_frontend_rng_state', 'sgb_frontend_h2d_bytes',
           'sgb_rng_draw', 'sgb_smooth_contour']


def lib_path():
    if os.environ.get('SGB_LIB_PATH'):      # an explicitly chosen build of the same library (A/B runs)
        return os.environ['SGB_LIB_PATH']
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), 'libsoundgen_b200.so')


_lib = None


def load():
    """Loads libsoundgen_b200.so.  There is no fallback: a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise RuntimeError('libsoundgen_b200.so is not built (%s); run '
                           '`python -c "import __graft_entry__ as g; g.build()"`' % p)
    L = C.CDLL(p)
    vp = C.c_void_p
    L.sgb_version.restype = C.c_int
    L.sgb_last_error.restype = C.c_char_p
    L.sgb_device_count.restype = C.c_int
    L.sgb_set_device.argtypes = [C.c_int]
    L.sgb_pin.argtypes = [vp, i64]
    L.sgb_device_pci_bus_id.argtypes = [C.c_int, C.c_char_p, C.c_int]
    L.sgb_unpin.argtypes = [vp]
    L.sgb_measure_fp32_peak.argtypes = [C.POINTER(f64)]
    L.sgb_batch_create.argtypes = [C.POINTER(vp)]
    L.sgb_batch_destroy.argtypes = [vp]
    L.sgb_batch_destroy.restype = None
    L.sgb_batch_upload.argtypes = [vp, C.POINTER(BatchDesc)]
    L.sgb_batch_run.argtypes = [vp, C.POINTER(RunInfo)]
    L.sgb_batch_lengths.argtypes = [vp, vp]
    L.sgb_batch_fetch_f32.argtypes = [vp, vp, i64]
    L.sgb_batch_fetch_f64.argtypes = [vp, vp, i64]
    L.sgb_batch_fetch_pcm16.argtypes = [vp, vp, i64]
    L.sgb_batch_status.argtypes = [vp, vp]
    L.sgb_batch_export.argtypes = [vp, C.POINTER(DeviceOut)]
    L.sgb_rows_export.argtypes = [i32, vp, vp, vp, i32, C.POINTER(DeviceOut)]
    L.sgb_spec_frames.argtypes = [i64, i32, f64]
    L.sgb_spec_frames.restype = i64
    L.sgb_batch_spectrogram.argtypes = [vp, C.POINTER(SpecParams), C.POINTER(DeviceOut)]
    L.sgb_rows_spectrogram.argtypes = [i32, vp, vp, vp, i32, C.POINTER(SpecParams), C.POINTER(DeviceOut)]
    L.sgb_rows_compare.argtypes = [i32, vp, i64, vp, i64, vp, vp, vp, vp, i32, C.POINTER(CompareParams), vp, i64, vp]
    L.sgb_param_range.argtypes = [C.c_char_p, vp]
    L.sgb_batch_syllable_len.argtypes = [vp, i32, C.POINTER(i64)]
    L.sgb_batch_syllable_fetch.argtypes = [vp, i32, vp, i64]
    L.sgb_batch_noise_fetch.argtypes = [vp, i32, vp, i64]
    L.sgb_batch_artefacts.argtypes = [vp, i32, C.POINTER(SylArtefacts)]
    L.sgb_batch_artefact_ints.argtypes = [vp, i32, C.c_int, vp, i32]
    L.sgb_batch_pitch_per_gc.argtypes = [vp, i32, vp, i32]
    L.sgb_batch_checksums.argtypes = [vp, vp, i32]
    L.sgb_batch_debug_state.argtypes = [vp, vp, i32]
    L.sgb_get_rolloff.argtypes = [vp, i32, i32, vp, i32, vp, i32, vp, i32, f64, f64, f64, f64,
                                  f64, f64, vp, C.POINTER(i32)]
    L.sgb_get_spectral_envelope.argtypes = [i32, i32, C.POINTER(Envelope), vp, vp, vp, vp]
    L.sgb_filter_len.argtypes = [i64, i32, f64]
    L.sgb_filter_len.restype = i64
    L.sgb_filter.argtypes = [vp, i64, vp, i32, i32, f64, vp, i64]
    L.sgb_batch_run_begin.argtypes = [vp]
    L.sgb_batch_run_finish.argtypes = [vp, C.POINTER(RunInfo)]
    L.sgb_batch_bout_geometry.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.sgb_batch_set_tracks.argtypes = [vp, i32, vp, i32, i32]
    L.sgb_batch_z_used.argtypes = [vp, vp]
    L.sgb_abi_sizes.argtypes = [vp, i32]
    L.sgb_frontend_create.argtypes = [C.POINTER(vp), i32]
    L.sgb_frontend_destroy.argtypes = [vp]
    L.sgb_frontend_destroy.restype = None
    L.sgb_frontend_add.argtypes = [vp, C.POINTER(SoundgenArgs)]
    L.sgb_frontend_add_seeded.argtypes = [vp, C.POINTER(SoundgenArgs), vp, i32]
    L.sgb_frontend_add_many.argtypes = [vp, vp, i32]
    L.sgb_frontend_clear.argtypes = [vp]
    L.sgb_synth_min_rows_set.argtypes = [i32]
    L.sgb_host_set_threads.argtypes = [i32]
    L.sgb_frontend_round_begin.argtypes = [vp, C.POINTER(BatchDesc), C.POINTER(i32)]
    L.sgb_frontend_resolve.argtypes = [vp, vp]
    L.sgb_frontend_round_end.argtypes = [vp, vp]
    L.sgb_frontend_round_calls.argtypes = [vp, vp]
    L.sgb_frontend_status.argtypes = [vp, vp]
    L.sgb_frontend_warnings.argtypes = [vp, i32]
    L.sgb_frontend_warnings.restype = C.c_char_p
    L.sgb_frontend_rng_state.argtypes = [vp, i32, vp]
    L.sgb_frontend_h2d_bytes.argtypes = [vp]
    L.sgb_frontend_h2d_bytes.restype = i64
    L.sgb_rng_draw.argtypes = [C.c_uint32, i32, f64, f64, i32, vp, i32]
    L.sgb_smooth_contour.argtypes = [vp, vp, i32, i32, f64, i32, f64, i32, f64, i32, i32, vp]
    sizes = (i32 * 12)()
    L.sgb_abi_sizes(sizes, 12)
    mine = [C.sizeof(t) for t in (Syllable, Envelope, Noise, Bout, Call, FormantRef, BatchDesc, RunInfo, SoundgenArgs,
                                  DeviceOut, SpecParams, CompareParams)]
    if list(sizes) != mine:
        raise RuntimeError('ctypes mirror out of date: library struct sizes %s, mirror %s' % (list(sizes), mine))
    _lib = L
    return L
