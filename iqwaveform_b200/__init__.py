"""iqwaveform_b200 -- B200-native spectral-analysis hot path of dgkuester/iqwaveform.

Drop-in (same names, arguments, error behaviour) for

    iqwaveform.fourier.stft / spectrogram / power_spectral_density (= persistence_spectrum)
    iqwaveform.power_analysis.iq_to_bin_power
    iqwaveform.fourier.upfirdn (scipy.signal.upfirdn semantics, zero padding)
    iqwaveform.fourier.oaconvolve (scipy.signal.oaconvolve semantics, one convolved axis)

backed by hand-written sm_100a CUDA kernels behind the C-ABI in ``include/iqw_b200.h``.
Importing the package loads ``libiqw_b200.so`` and fails loudly when it is missing: there is no
CPU fallback.
"""
from . import _lib  # noqa: F401  (raises ImportError when the CUDA library is absent)
from . import fourier, power_analysis, distributed, util, io
from .util import Domain, set_input_domain, get_input_domain
from .fourier import (fft, ifft, zero_stft_by_freq, stft, istft, ola_filter, oaresample, upfirdn, oaconvolve, iq_to_stft_spectrogram, channelize_power, spectrogram, power_spectral_density, persistence_spectrum, fftfreq,
                      get_window, equivalent_noise_bandwidth, time_statistics, GraphedCall)
from .power_analysis import (iq_to_bin_power, iq_to_cyclic_power, powtodB, dBtopow, envtopow, envtodB, dBlinmean, dBlinsum,
                             sample_ccdf)
from .util import histogram_last_axis, isroundmod, to_blocks
from ._plan import find_window_param_from_enbw
from .io import read_sigmf, read_sigmf_metadata, waveform_to_frame, persistence_spectrum_from_sigmf

__version__ = '0.2.0'
__all__ = ['GraphedCall', 'fourier', 'power_analysis', 'distributed', 'util', 'io', 'read_sigmf', 'read_sigmf_metadata', 'waveform_to_frame',
           'persistence_spectrum_from_sigmf', 'Domain', 'set_input_domain', 'get_input_domain', 'fft', 'ifft', 'zero_stft_by_freq', 'stft', 'istft', 'ola_filter', 'oaresample', 'upfirdn', 'oaconvolve', 'iq_to_stft_spectrogram', 'channelize_power', 'sample_ccdf', 'histogram_last_axis', 'isroundmod', 'to_blocks', 'find_window_param_from_enbw', 'spectrogram', 'power_spectral_density',
           'persistence_spectrum', 'fftfreq', 'get_window', 'equivalent_noise_bandwidth',
           'time_statistics', 'iq_to_bin_power', 'iq_to_cyclic_power', 'powtodB', 'dBtopow', 'envtopow', 'envtodB', 'dBlinmean',
           'dBlinsum']
