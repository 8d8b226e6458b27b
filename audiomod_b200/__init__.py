"""audiomod_b200: B200-native phase-vocoder path of tangkk/audiomod behind the reference's modbase API."""
from .phasevocoder import (CONSTANT, FORMANT_CEPSTRAL, FORMANT_PRESERVE, GENDER_CEPSTRAL, GENDER_CHANGE, INT_RATIO, NORMAL_PV, NORMAL_SHIFT, NORMAL_STRETCH,
                           PHASE_LOCKED, ROBOTIC, VOCODER_CHORD, VOCODER_ROSENBERG, WHISPER, HostBuffer, PhaseVocoderBatch,
                           PhaseVocoderMultiBatch, biquad_design, describe, equalizer_chain, kweighting_design, plan_counts, phasevocoder, run_wav_files, shard_streams)
from ._lib import F32, S16, PvgpuError

__all__ = ["phasevocoder", "PhaseVocoderBatch", "PhaseVocoderMultiBatch", "HostBuffer", "shard_streams", "run_wav_files", "equalizer_chain", "biquad_design", "kweighting_design", "describe", "plan_counts", "PvgpuError", "F32", "S16", "CONSTANT", "NORMAL_SHIFT", "GENDER_CHANGE",
           "FORMANT_PRESERVE", "GENDER_CEPSTRAL", "FORMANT_CEPSTRAL", "VOCODER_ROSENBERG", "VOCODER_CHORD", "NORMAL_STRETCH", "ROBOTIC", "WHISPER", "NORMAL_PV",
           "PHASE_LOCKED", "INT_RATIO"]
