"""soundgen_beta_b200 -- B200-native source-filter synthesis path of soundgen behind the
reference's own function names.  All compute goes through libsoundgen_b200.so (CUDA,
sm_100a); importing this package never falls back to a CPU implementation."""
from .api import (ArgArray, Batch, BatchBuilder, FrontEnd, run_rounds, PipelinedBatches, SoundgenError, filter_sound, generateHarmonics, generateNoise,
                  getRolloff, getSpectralEnvelope, mel_filterbank, pin_desc, rows_export, rows_spectrogram, soundgen,
                  soundgen_batch, soundgen_batch_device, spectrogram_device)

__all__ = ['ArgArray', 'Batch', 'BatchBuilder', 'FrontEnd', 'run_rounds', 'PipelinedBatches', 'SoundgenError', 'filter_sound', 'generateHarmonics', 'generateNoise',
           'getRolloff', 'getSpectralEnvelope', 'mel_filterbank', 'pin_desc', 'rows_export', 'rows_spectrogram', 'soundgen',
           'soundgen_batch', 'soundgen_batch_device', 'spectrogram_device']
