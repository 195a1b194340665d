"""ultrazoom_b200 -- B200-native MewZoom.upscale hot path (drop-in for ``ultrazoom`` 0.2.x inference).

    from ultrazoom_b200.model import MewZoom
    from ultrazoom_b200.control import ControlVector
"""
from .control import ControlVector  # noqa: F401
from .model import MewZoom, ONNXModel, Yuv420  # noqa: F401

MODEL_CONFIGS = {
    # reference README.md:35-42 (channels, encoder layers); hidden_ratio 2 = pretrain.py:74 default
    "MewZoom-2X": dict(upscale_ratio=2, num_channels=48, hidden_ratio=2, num_encoder_layers=20, control_features=0),
    "MewZoom-3X": dict(upscale_ratio=3, num_channels=54, hidden_ratio=2, num_encoder_layers=30, control_features=0),
    "MewZoom-4X": dict(upscale_ratio=4, num_channels=96, hidden_ratio=2, num_encoder_layers=40, control_features=0),
    "MewZoom-2X-Ctrl": dict(upscale_ratio=2, num_channels=48, hidden_ratio=2, num_encoder_layers=20, control_features=3),
    "MewZoom-3X-Ctrl": dict(upscale_ratio=3, num_channels=54, hidden_ratio=2, num_encoder_layers=30, control_features=3),
    "MewZoom-4X-Ctrl": dict(upscale_ratio=4, num_channels=96, hidden_ratio=2, num_encoder_layers=40, control_features=3),
}

__version__ = "0.1.0"
