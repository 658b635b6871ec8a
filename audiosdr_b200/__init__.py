"""audiosdr_b200 -- B200-native batched implementation of AudioSDR's per-block receiver chain.

The hot path `AudioSDR::update()` (reference SRC/AudioSDRlib/AudioSDR.cpp:39-168) is implemented behind the C ABI of
include/sdr_batch.h; the blocks either side of it (SURVEY 8f: AudioSDRpreProcessor, AudioIQgenerator) behind
include/sdr_aux.h (`PreProcessorBatch`, `IQGeneratorBatch`).  `SdrBatch` mirrors the reference class's setter names with a
channel selector.  `GraphBatch` (include/sdr_graph.h) streams the sketch's whole graph -- front, grabber tap, receiver --
from host memory in one ticketed call.  The CUDA library is mandatory: importing works without it (so that the CPU-only test
tier can import the package), but constructing an SdrBatch raises unless libsdr_batch.so loads and a
CUDA device accepts the sm_100a kernel image.  There is no CPU fallback.
"""
from .api import (AGC_FAST, AGC_MEDIUM, AGC_OFF, AGC_SLOW, AM, AUDIO_2100, AUDIO_2300, AUDIO_2500, AUDIO_2700,
                  AUDIO_2900, AUDIO_3100, AUDIO_3300, AUDIO_AM, AUDIO_BYPASS, AUDIO_CW, AUDIO_WSPR, BS_AGC_ACTIVE,
                  BS_AGC_GAIN, BS_AM_CARRIER, BS_FIELDS, BS_NAMES, BS_NB_AVERAGE, BS_NB_DETECTED, BS_SAM_FREQUENCY,
                  BS_SAM_LOCKED, CW_LSB, CW_USB, FMT_F32, FMT_I16, LSB, SAM, SETTERS, USB, WSPR, ChannelStatus, SdrBatch,
                  SdrError, block_status_fields, lib_path, load_library)
from .aux import AuxError, GrabberBatch, IQGeneratorBatch, PreProcessorBatch, WaterfallBatch
from .build import build_aux_library, build_graph_library, build_library
from .graph import GraphBatch, GraphError

__all__ = [n for n in dir() if not n.startswith("_")]
