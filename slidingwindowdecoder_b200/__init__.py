"""B200-native batched window decoders with the SlidingWindowDecoder Python API."""
from .decoders import bpgdg_decoder, bpgd_decoder, osd_window, BpOsdDecoder, bp4_osd  # noqa: F401
from .simulation import CodeCapacitySampler, CircuitNoiseSampler, depolarizing_noise_decoding  # noqa: F401
from .drivers import circuit_erasure_decoding, circuit_soft_readout_decoding  # noqa: F401
from .dem import gaussian_readout  # noqa: F401

__version__ = "0.1.0"
