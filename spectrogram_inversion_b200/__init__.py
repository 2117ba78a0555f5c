"""spectrogram_inversion_b200 -- B200-native (sm_100a) drop-in for the iterative STFT/ISTFT
phase-retrieval hot path of torch_specinv 0.2.1 (griffin_lim, RTISI_LA, ADMM, sc/snr/ser)."""
from . import methods, metrics, torchaudio_compat
from .methods import ADMM, L_BFGS, RTISI_LA, griffin_lim, phase_init
from .metrics import sc, ser, snr, spectral_convergence
from .pghi import pghi
from .streaming import PGHIStream, RTISIStream

__version__ = "0.1.0"
__all__ = ["griffin_lim", "RTISI_LA", "RTISIStream", "PGHIStream", "ADMM", "L_BFGS", "phase_init", "pghi", "sc", "snr", "ser", "spectral_convergence",
           "methods", "metrics", "torchaudio_compat"]
