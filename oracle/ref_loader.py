"""Import the reference's OWN hot-path modules from the reference checkout (POSEDIFF_REFERENCE_ROOT).

TEST INFRASTRUCTURE.  Where the checkout is absent, the same unmodified modules are imported from oracle/_ref (installed
there by oracle/install_reference.py during `build()`).  Used by `oracle/make_golden.py` (fixture generation) and by
`bench.py --impl reference` / the `cpu_baseline` leg, which time the oracle port when neither is present.
pytorch3d and hydra are not installed here; `oracle/shims/` restates the handful of symbols
the reference imports (SURVEY.md §8c).  Nothing is copied: the modules are imported in place.
"""
from __future__ import annotations

import os
import sys
from types import SimpleNamespace

REFERENCE_ROOT = os.environ.get("POSEDIFF_REFERENCE_ROOT", "/root/reference")
_SHIMS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "shims")
# the unmodified `models` / `util` packages installed by oracle/install_reference.py (git-ignored build output)
INSTALLED_ROOT = os.environ.get("POSEDIFF_INSTALLED_REFERENCE", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))

TRANSFORMER_CFG = dict(
    _target_="models.TransformerEncoderWrapper",
    d_model=512,
    nhead=4,
    dim_feedforward=1024,
    num_encoder_layers=8,
    dropout=0.1,
    batch_first=True,
    norm_first=True,
)  # cfgs/default.yaml:27-35


def reference_path() -> str | None:
    """Directory that holds the reference's `models` and `util` packages: the reference checkout when present, else the
    copy installed into oracle/_ref, else None."""
    src = os.path.join(REFERENCE_ROOT, "pose_diffusion")
    if os.path.isdir(os.path.join(src, "models")):
        return src
    if os.path.isdir(os.path.join(INSTALLED_ROOT, "models")) and os.path.isdir(os.path.join(INSTALLED_ROOT, "util")):
        return INSTALLED_ROOT
    return None


def reference_available() -> bool:
    return reference_path() is not None


def load_reference() -> SimpleNamespace:
    """Returns namespace(Denoiser, GaussianDiffusion, geometry_guided_sampling, GGS_optimize,
    compute_sampson_distance, pose_encoding_to_camera, get_fundamental_matrices, to_attr)."""
    where = reference_path()
    if where is None:
        raise FileNotFoundError(f"reference modules not found under {REFERENCE_ROOT} or {INSTALLED_ROOT}")
    for path in (where, _SHIMS):
        if path not in sys.path:
            sys.path.insert(0, path)
    import hydra.utils as hydra_utils  # the shim
    import models  # reference package: pose_diffusion/models/__init__.py
    from util import camera_transform, geometry_guided_sampling as ggs, get_fundamental_matrix

    return SimpleNamespace(
        Denoiser=models.Denoiser,
        GaussianDiffusion=models.GaussianDiffusion,
        geometry_guided_sampling=ggs.geometry_guided_sampling,
        GGS_optimize=ggs.GGS_optimize,
        compute_sampson_distance=ggs.compute_sampson_distance,
        pose_encoding_to_camera=camera_transform.pose_encoding_to_camera,
        get_fundamental_matrices=get_fundamental_matrix.get_fundamental_matrices,
        to_attr=hydra_utils.to_attr,
    )


def build_reference_sampler(ref: SimpleNamespace, denoiser_state: dict):
    """Reference GaussianDiffusion with a reference Denoiser attached (pose_diffusion_model.py:57-61),
    weights loaded strictly from `denoiser_state` (keys relative to `diffuser.model.`)."""
    denoiser = ref.Denoiser(TRANSFORMER=ref.to_attr(TRANSFORMER_CFG))
    denoiser.load_state_dict(denoiser_state, strict=True)
    diffuser = ref.GaussianDiffusion(beta_schedule="custom")
    diffuser.model = denoiser
    return diffuser.eval()
