"""comfy_rvc_b200 — B200-native (sm_100a) RVC synthesis hot path behind the reference's Python API."""
from .config import NAMED_CONFIGS, SynthConfig  # noqa: F401
from .synthesizer import (SynthesizerB200, SynthesizerTrnMs256NSFsid, SynthesizerTrnMs768NSFsid,  # noqa: F401
                          SynthesizerTrnMs256NSFsid_nono, SynthesizerTrnMs768NSFsid_nono)

from .index import IndexIVFFlatB200  # noqa: F401
from .pipeline import VC, FeatureExtractor, PipelineConfig, get_vc  # noqa: F401
from .hubert import HubertB200  # noqa: F401
from .rmvpe import RMVPE  # noqa: F401
from . import crepe  # noqa: F401

__all__ = ["crepe", "HubertB200", "IndexIVFFlatB200", "RMVPE", "VC", "FeatureExtractor", "PipelineConfig", "get_vc", "SynthesizerTrnMs256NSFsid", "SynthesizerTrnMs768NSFsid", "SynthesizerTrnMs256NSFsid_nono", "SynthesizerTrnMs768NSFsid_nono", "SynthesizerB200", "SynthConfig", "NAMED_CONFIGS"]
