"""B200-native (sm_100a) mastering DSP chain behind the settings dict and entry points of
theouterlimitz/Audio-Mastering-Engine (audio_mastering_engine.py:94, :171).  See DESIGN.md."""
from .engine import (EQ_PRESETS, MasterPlan, bind_host_to_gpu_numa, limit_device, master, measure_loudness, process_audio,
                     process_audio_with_ffmpeg_pipeline, read_wav, release_cached_memory, write_wav)
from ._lib import AmeError

__all__ = ["EQ_PRESETS", "MasterPlan", "master", "process_audio", "process_audio_with_ffmpeg_pipeline",
           "read_wav", "write_wav", "AmeError", "bind_host_to_gpu_numa", "release_cached_memory", "limit_device",
           "measure_loudness"]
