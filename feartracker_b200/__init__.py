"""feartracker_b200 -- B200-native (sm_100a) implementation of the FEAR-XS per-frame inference hot
path behind the reference's FEARNet / FEARTracker API.  See DESIGN.md."""
from .constants import TARGET_CLASSIFICATION_KEY, TARGET_REGRESSION_LABEL_KEY  # noqa: F401
from .fear_net import FEARNet  # noqa: F401
from .box_coder import FEARBoxCoder, TrackerDecodeResult  # noqa: F401
from .tracker import FEARTracker, Tracker, TrackingState  # noqa: F401
from .multi_tracker import FEARMultiTracker  # noqa: F401

FEAR_XS_MODEL_KWARGS = dict(  # reference model_training/config/model/fear.yaml
    backbone="custom_fbnet", img_size=256, pretrained=True, stride=2, conv_block="sep_conv", towernum=2, mobile=True,
    max_layer=4, crop_template_features=False,
)
FEAR_XS_TRACKER_KWARGS = dict(  # reference model_training/config/tracker/siam_tracker.yaml
    penalty_k=0.062, window_influence=0.38, lr=0.765, windowing="cosine", total_stride=16, score_size=16, ratio=0.94,
    stride=2, bbox_ratio=0.5, template_bbox_offset=0.2, search_context=2, instance_size=256, template_size=128,
)


def load_from_lighting(model, checkpoint_path: str, map_location=None, strict: bool = True):
    """Load a Lightning checkpoint the way the reference does (model_training/utils/torch.py:11-24): an int
    ``map_location`` means ``cuda:<n>``; keys under ``model.`` are kept with the prefix stripped; ``strict=True`` is a
    strict ``load_state_dict``; ``strict=False`` has pytorch_toolbelt ``transfer_weights`` semantics -- every tensor
    is loaded on its own and the ones whose name or shape does not match are skipped instead of raising."""
    import torch

    if type(map_location) is int:
        map_location = f"cuda:{map_location}"
    ckpt = torch.load(checkpoint_path, map_location=map_location, weights_only=True)
    sd = {k[len("model."):]: v for k, v in ckpt["state_dict"].items() if k.startswith("model.")}
    if strict:
        model.load_state_dict(sd, strict=True)
        return model
    skipped = []
    for name, value in sd.items():
        try:
            model.load_state_dict({name: value}, strict=False)
        except Exception:  # size mismatch for this tensor: skip it, like transfer_weights
            skipped.append(name)
    if skipped:
        import warnings

        warnings.warn(f"load_from_lighting(strict=False): skipped {len(skipped)} tensors with mismatching shapes "
                      f"(first: {skipped[0]})")
    return model
