"""ddsp_b200 - B200-native (sm_100a) Harmonic + FilteredNoise DDSP decoder.

Drop-in for the signal-generation layer of magenta/ddsp: `Processor`,
`ProcessorGroup`, `Harmonic`, `FilteredNoise`, `Add` with the reference's API,
backed by hand-written CUDA kernels behind a ctypes C ABI (include/ddsp_b200.h).
"""
from ddsp_b200 import _lib
from ddsp_b200 import core
from ddsp_b200 import dags
from ddsp_b200 import effects
from ddsp_b200 import host
from ddsp_b200 import processors
from ddsp_b200 import synths
from ddsp_b200.effects import FIRFilter, FilteredNoiseReverb, ModDelay, Reverb
from ddsp_b200.host import HostDecoder
from ddsp_b200.processors import Add, Processor, ProcessorGroup
from ddsp_b200.synths import FilteredNoise, Harmonic, Sinusoidal, Wavetable

__version__ = '0.1.0'
