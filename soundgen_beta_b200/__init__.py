"""soundgen_beta_b200 -- B200-native source-filter synthesis path of soundgen behind the
reference's own function names.  All compute goes through libsoundgen_b200.so (CUDA,
sm_100a); importing this package never falls back to a CPU implementation."""
from .api import (ArgArray, Batch, BatchBuilder, FrontEnd, run_rounds, PipelinedBatches, SoundgenError, compare_spectrograms,
                  dct_matrix, f0_frames_device, filter_sound, generateHarmonics, generateNoise, getRolloff, getSpectralEnvelope,
                  match_pars, mel_filterbank, mfcc_device, param_range, pin_desc, rows_cepstra, rows_export,
                  rows_f0_frames, rows_spectrogram, soundgen, soundgen_batch, soundgen_batch_device, spectrogram_device, wiggle_pars)

__all__ = ['ArgArray', 'Batch', 'BatchBuilder', 'FrontEnd', 'run_rounds', 'PipelinedBatches', 'SoundgenError',
           'compare_spectrograms', 'dct_matrix', 'f0_frames_device', 'filter_sound', 'generateHarmonics', 'generateNoise', 'getRolloff',
           'getSpectralEnvelope', 'match_pars', 'mel_filterbank', 'mfcc_device', 'param_range', 'pin_desc',
           'rows_cepstra', 'rows_export', 'rows_f0_frames', 'rows_spectrogram', 'soundgen', 'soundgen_batch', 'soundgen_batch_device',
           'spectrogram_device', 'wiggle_pars']
