"""Golden-case catalogue shared by the fixture generator and the parity tests.

TEST INFRASTRUCTURE.  Each case names a transform spec (class name + kwargs,
the reference's own spelling), a global torch seed, and how to synthesise the
inputs.  ``tests/golden/generate.py`` runs the real reference on these and
stores outputs + sampled params; the tests replay the stored params through
the oracle (CPU) and the CUDA path (GPU) and compare.
"""

from __future__ import annotations

import numpy as np
import torch


def _affine(spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0), tilt=0.0):
    """Voxel->world 4x4 (float64) with optional small in-plane rotation."""
    m = np.eye(4, dtype=np.float64)
    c, s = np.cos(tilt), np.sin(tilt)
    direction = np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    m[:3, :3] = direction * np.asarray(spacing, dtype=np.float64)
    m[:3, 3] = origin
    return m


def scalar_volume(shape, seed, channels=1, shift=0.0):
    gen = torch.Generator().manual_seed(seed)
    return torch.rand((channels, *shape), generator=gen) - shift


def label_volume(shape, dtype=torch.int16, channels=1):
    """Concentric boxes with labels 0..4 (deterministic, no RNG)."""
    i, j, k = (torch.arange(n, dtype=torch.float32) for n in shape)
    ci, cj, ck = ((n - 1) / 2 for n in shape)
    di = (i - ci).abs()[:, None, None] / max(shape[0], 1)
    dj = (j - cj).abs()[None, :, None] / max(shape[1], 1)
    dk = (k - ck).abs()[None, None, :] / max(shape[2], 1)
    d = torch.maximum(torch.maximum(di, dj), dk)  # in [0, 0.5]
    lab = (4 - torch.clamp((d * 10).floor(), max=4)).to(dtype)
    return lab[None].repeat(channels, 1, 1, 1).contiguous()


def build_inputs(case):
    shape = tuple(case["shape"])
    affine = _affine(
        case.get("spacing", (1.0, 1.0, 1.0)),
        case.get("origin", (0.0, 0.0, 0.0)),
        case.get("tilt", 0.0),
    )
    subjects = []
    for b in range(case["batch"]):
        sub = {}
        for name, kind in case["images"].items():
            if kind == "scalar":
                seed = 1000 + b + 97 * len(sub)
                tensor = scalar_volume(
                    shape,
                    seed,
                    channels=case.get("channels", 1),
                    shift=case.get("shift", 0.0),
                )
                sub[name] = ("scalar", tensor, affine)
            else:
                dtype = getattr(torch, kind)
                sub[name] = ("label", label_volume(shape, dtype), affine)
        subjects.append(sub)
    return {"subjects": subjects}


_AFF = {"scales": (0.9, 1.1), "degrees": (-10, 10), "translation": (-3, 3)}

CASES = [
    # BASELINE.json configs[0]: correctness plumbing case.
    dict(name="config1_affine_deg10_64", seed=1234, shape=(64, 64, 64), batch=1,
         images={"t1": "scalar"}, transform=("Affine", {"degrees": 10})),
    dict(name="affine_b1_label", seed=11, shape=(20, 17, 13), batch=1,
         images={"t1": "scalar", "seg": "int16"}, transform=("Affine", _AFF)),
    dict(name="affine_b3_aniso", seed=12, shape=(18, 15, 12), batch=3,
         spacing=(0.8, 1.1, 2.0), origin=(-7.0, 3.5, 10.0), tilt=0.1,
         images={"t1": "scalar", "seg": "uint8"}, transform=("Affine", _AFF)),
    dict(name="affine_fill_zero", seed=13, shape=(16, 14, 12), batch=2,
         images={"t1": "scalar"},
         transform=("Affine", {**_AFF, "default_pad_value": 0.0})),
    dict(name="affine_fill_number", seed=14, shape=(16, 14, 12), batch=2,
         images={"t1": "scalar", "seg": "int32"},
         transform=("Affine", {**_AFF, "default_pad_value": -1.5,
                               "default_pad_label": 7})),
    dict(name="affine_fill_mean", seed=24, shape=(16, 14, 12), batch=2, channels=2,
         images={"t1": "scalar"}, transform=("Affine", {**_AFF, "default_pad_value": "mean"})),
    dict(name="affine_fill_otsu", seed=25, shape=(16, 14, 12), batch=2, channels=2,
         images={"t1": "scalar"}, transform=("Affine", {**_AFF, "default_pad_value": "otsu"})),
    dict(name="affine_nearest_image", seed=15, shape=(16, 14, 12), batch=2,
         images={"t1": "scalar"},
         transform=("Affine", {**_AFF, "image_interpolation": "nearest"})),
    dict(name="affine_gated", seed=16, shape=(12, 12, 10), batch=5,
         images={"t1": "scalar", "seg": "int64"},
         transform=("Affine", {**_AFF, "p": 0.5})),
    dict(name="affine_multichannel", seed=17, shape=(12, 11, 10), batch=2,
         channels=3, shift=0.4, images={"t1": "scalar"},
         transform=("Affine", _AFF)),
    dict(name="elastic_b1", seed=21, shape=(24, 20, 16), batch=1,
         images={"t1": "scalar", "seg": "int16"},
         transform=("ElasticDeformation", {"max_displacement": 2.0})),
    dict(name="elastic_b3_aniso", seed=22, shape=(20, 18, 14), batch=3,
         spacing=(0.8, 1.1, 2.0), origin=(2.0, -3.0, 1.0),
         images={"t1": "scalar", "seg": "int32"},
         transform=("ElasticDeformation",
                    {"max_displacement": (1.0, 3.0),
                     "num_control_points": (5, 6, 7), "locked_borders": 1})),
    dict(name="spatial_affine_first", seed=23, shape=(18, 16, 14), batch=2,
         spacing=(1.2, 0.9, 1.5),
         images={"t1": "scalar", "seg": "uint8"},
         transform=("Spatial", {**_AFF, "max_displacement": (1.0, 2.5),
                                "num_control_points": 6})),
    dict(name="spatial_elastic_first", seed=24, shape=(18, 16, 14), batch=2,
         spacing=(1.2, 0.9, 1.5),
         images={"t1": "scalar", "seg": "uint8"},
         transform=("Spatial", {**_AFF, "max_displacement": (1.0, 2.5),
                                "num_control_points": 6,
                                "affine_first": False})),
    dict(name="spatial_shared", seed=25, shape=(14, 13, 12), batch=3,
         images={"t1": "scalar"},
         transform=("Spatial", {**_AFF, "max_displacement": 1.5,
                                "per_instance": False})),
    dict(name="bias_b1", seed=31, shape=(20, 17, 13), batch=1,
         images={"t1": "scalar", "seg": "int16"},
         transform=("BiasField", {})),
    dict(name="bias_b3_gated", seed=32, shape=(16, 14, 12), batch=4,
         channels=2, images={"t1": "scalar"},
         transform=("BiasField", {"std": (0.1, 0.6), "p": 0.6})),
    dict(name="bias_shared", seed=33, shape=(16, 14, 12), batch=3,
         images={"t1": "scalar"},
         transform=("BiasField", {"per_instance": False})),
    dict(name="bias_large_scale", seed=34, shape=(40, 30, 20), batch=2,
         images={"t1": "scalar"},
         transform=("BiasField", {"scale": 0.3})),
    dict(name="blur_b1", seed=41, shape=(20, 17, 13), batch=1,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Blur", {"std": (0.5, 2.0)})),
    dict(name="blur_b3_aniso", seed=42, shape=(18, 15, 12), batch=3,
         spacing=(0.8, 1.1, 2.0), images={"t1": "scalar"},
         transform=("Blur", {"std": (0.0, 2.0)})),
    dict(name="blur_shared", seed=43, shape=(16, 14, 12), batch=3, channels=2,
         images={"t1": "scalar"},
         transform=("Blur", {"std": (0.5, 2.0), "per_instance": False})),
    dict(name="blur_gated", seed=44, shape=(12, 12, 10), batch=5,
         images={"t1": "scalar"},
         transform=("Blur", {"std": (0.5, 2.0), "p": 0.5})),
    dict(name="blur_one_axis", seed=45, shape=(12, 12, 10), batch=1,
         images={"t1": "scalar"},
         transform=("Blur", {"std": (0.0, 1.3, 0.0)})),
    dict(name="noise_b1", seed=51, shape=(20, 17, 13), batch=1,
         images={"t1": "scalar", "seg": "int16"}, transform=("Noise", {})),
    dict(name="noise_b3_two_images", seed=52, shape=(16, 16, 16), batch=3,
         images={"t1": "scalar", "t2": "scalar"},
         transform=("Noise", {"mean": (-0.1, 0.1), "std": (0.0, 0.25)})),
    dict(name="noise_ragged_tail", seed=53, shape=(5, 7, 3), batch=2,
         images={"t1": "scalar", "t2": "scalar"},
         transform=("Noise", {"std": (0.0, 0.25)})),
    dict(name="noise_rician_gated", seed=54, shape=(12, 12, 10), batch=5,
         shift=0.3, images={"t1": "scalar"},
         transform=("Noise", {"std": (0.05, 0.25), "rician": True, "p": 0.5})),
    dict(name="gamma_b1", seed=61, shape=(20, 17, 13), batch=1, shift=0.3,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Gamma", {"log_gamma": (-0.3, 0.3)})),
    dict(name="gamma_b4_gated", seed=62, shape=(12, 12, 10), batch=4,
         shift=0.3, images={"t1": "scalar"},
         transform=("Gamma", {"log_gamma": (-0.3, 0.3), "p": 0.7})),
    dict(name="compose_config2_b2", seed=71, shape=(24, 20, 16), batch=2,
         images={"t1": "scalar", "seg": "int16"},
         transform=[("Affine", {"scales": (0.9, 1.1), "degrees": (-10, 10)}),
                    ("ElasticDeformation", {"max_displacement": 2.0})]),
    dict(name="compose_full_b2", seed=72, shape=(24, 20, 16), batch=2,
         images={"t1": "scalar", "seg": "int16"},
         transform=[("Affine", {"scales": (0.9, 1.1), "degrees": (-10, 10)}),
                    ("ElasticDeformation", {"max_displacement": 2.0}),
                    ("BiasField", {}),
                    ("Blur", {"std": (0.0, 2.0)}),
                    ("Noise", {"std": (0.0, 0.25)}),
                    ("Gamma", {"log_gamma": (-0.3, 0.3)})]),
    dict(name="compose_full_b1_48", seed=73, shape=(48, 48, 48), batch=1,
         images={"t1": "scalar"},
         transform=[("Affine", {"scales": (0.9, 1.1), "degrees": (-10, 10)}),
                    ("ElasticDeformation", {}),
                    ("BiasField", {}),
                    ("Blur", {"std": (0.0, 2.0)}),
                    ("Noise", {"std": (0.0, 0.25)}),
                    ("Gamma", {"log_gamma": (-0.3, 0.3)})]),
    # ---- K1 tile kernels (TMA boxes): K * element size a multiple of 16 bytes and at least one
    # full 16^3 output tile per axis, so most tiles walk the staged box instead of the general column
    dict(name="elastic_aniso_tiles", seed=131, shape=(40, 36, 48), batch=2,
         spacing=(0.8, 1.1, 2.0), origin=(2.0, -3.0, 1.0),
         images={"t1": "scalar", "seg": "uint8"},
         transform=("ElasticDeformation", {"max_displacement": (3.0, 5.0, 6.0),
                                           "num_control_points": (7, 6, 8)})),
    # control cells of 5.2 / 6.5 / 5.25 voxels, the densest grid whose every tile the bounds pre-pass
    # still accepts (it gives up beyond two cell crossings per 16-voxel tile axis): the walk changes
    # cell inside a 16-plane tile two or three times, sometimes between the planes of one pair
    dict(name="elastic_dense_grid_tiles", seed=132, shape=(48, 40, 64), batch=1,
         spacing=(1.0, 1.0, 2.0), images={"t1": "scalar", "seg": "int16"},
         transform=("ElasticDeformation", {"max_displacement": 1.5,
                                           "num_control_points": (10, 7, 13), "locked_borders": 0})),
    # half-voxel translations: fill decisions exactly on the mask threshold of 0.5
    dict(name="affine_half_voxel_fill", seed=133, shape=(40, 36, 48), batch=1, channels=2,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Affine", {"scales": (1.0, 1.0), "degrees": (0.0, 0.0),
                               "translation": (0.5, 0.5, -1.5, -1.5, 2.5, 2.5),
                               "default_pad_value": -1.0, "default_pad_label": 7})),
]

# ---- index-remap neighbours of the chain (SURVEY §8 f-3): Flip / Crop / Pad ----------
NEIGHBOUR_CASES = [
    dict(name="flip_b4_per_instance", seed=81, shape=(10, 12, 14), batch=4,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Flip", {"axes": (0, 1, 2), "flip_probability": 0.5})),
    dict(name="flip_gated_two_axes", seed=82, shape=(9, 8, 16), batch=5, channels=2,
         images={"t1": "scalar"}, transform=("Flip", {"axes": (0, 2), "p": 0.6})),
    dict(name="flip_shared", seed=83, shape=(8, 9, 10), batch=3,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Flip", {"axes": (1, 2), "flip_probability": 0.7, "per_instance": False})),
    dict(name="crop_aniso", seed=84, shape=(12, 13, 14), batch=2, spacing=(1.0, 1.5, 2.0),
         origin=(5.0, -3.0, 2.0), tilt=0.2, images={"t1": "scalar", "seg": "int16"},
         transform=("Crop", {"cropping": (1, 2, 3, 0, 2, 1)})),
    dict(name="pad_constant", seed=85, shape=(8, 9, 10), batch=2, spacing=(2.0, 1.0, 0.5),
         images={"t1": "scalar", "seg": "int16"},
         transform=("Pad", {"padding": (2, 1, 0, 3, 1, 2), "fill": 1.5})),
    dict(name="pad_reflect", seed=86, shape=(8, 9, 10), batch=2, images={"t1": "scalar"},
         transform=("Pad", {"padding": (3, 2, 1), "padding_mode": "reflect"})),
    dict(name="pad_replicate", seed=87, shape=(8, 9, 10), batch=1, images={"t1": "scalar", "seg": "int16"},
         transform=("Pad", {"padding": 4, "padding_mode": "replicate"})),
    dict(name="pad_circular", seed=88, shape=(8, 9, 10), batch=2, images={"t1": "scalar"},
         transform=("Pad", {"padding": (2, 3, 4, 5, 6, 7), "padding_mode": "circular"})),
    # whole-volume statistic per element (_padding.py:41-110)
    dict(name="pad_minimum", seed=90, shape=(8, 9, 10), batch=3, channels=2, shift=0.3,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Pad", {"padding": (2, 1, 0, 3, 1, 2), "padding_mode": "minimum"})),
    dict(name="pad_median", seed=91, shape=(9, 8, 11), batch=2, channels=2, shift=0.3,
         images={"t1": "scalar"}, transform=("Pad", {"padding": (1, 2, 3), "padding_mode": "median"})),
    dict(name="pad_mean", seed=92, shape=(8, 9, 10), batch=2, shift=0.3,
         images={"t1": "scalar"}, transform=("Pad", {"padding": 2, "padding_mode": "mean"})),
    dict(name="compose_flip_pad_affine_crop", seed=89, shape=(16, 16, 16), batch=2,
         images={"t1": "scalar", "seg": "int16"},
         transform=[("Flip", {"axes": (0, 1, 2), "flip_probability": 0.5}),
                    ("Pad", {"padding": (2, 2, 4)}),
                    ("Affine", {"scales": (0.9, 1.1), "degrees": (-10, 10)}),
                    ("Crop", {"cropping": (2, 2, 4)})]),
]

# transforms whose history holds derived records (CropOrPad leaves Pad + Crop + itself):
# checked through the public call only, never by replaying the stored history
CALL_CASES = [
    dict(name="croporpad_center", seed=91, shape=(14, 9, 12), batch=2, spacing=(1.0, 2.0, 1.5),
         images={"t1": "scalar", "seg": "int16"},
         transform=("CropOrPad", {"target_shape": (10, 12, 12)})),
    dict(name="croporpad_random_mm", seed=92, shape=(16, 10, 12), batch=2, spacing=(1.0, 2.0, 0.5),
         images={"t1": "scalar"},
         transform=("CropOrPad", {"target_shape": (12.0, 24.0, 4.0), "units": "mm", "location": "random",
                                  "padding_mode": "replicate"})),
    dict(name="croporpad_only_pad", seed=93, shape=(8, 12, 10), batch=1, images={"t1": "scalar", "seg": "int16"},
         transform=("CropOrPad", {"target_shape": (12, 8, None), "only_pad": True, "fill": 2.5})),
]

# ---- data-derived intensity maps (SURVEY §8 f-3): Standardize / Normalize ---------------------
# Their params hold statistics of batch element 0, so the host-params tests (CPU, kernels stubbed)
# do not cover them: tests/test_gpu_stats.py checks sampling + statistics + map on the GPU.
STAT_CASES = [
    dict(name="standardize_b2", seed=101, shape=(24, 20, 16), batch=2, shift=0.3,
         images={"t1": "scalar", "seg": "int16"}, transform=("Standardize", {})),
    dict(name="standardize_masked", seed=102, shape=(24, 20, 16), batch=2, channels=2,
         images={"t1": "scalar", "seg": "int16"}, transform=("Standardize", {"masking_method": "seg"})),
    dict(name="normalize_default_b2", seed=103, shape=(24, 20, 16), batch=2, shift=0.3,
         images={"t1": "scalar", "seg": "int16"}, transform=("Normalize", {})),
    dict(name="normalize_percentiles", seed=104, shape=(32, 28, 24), batch=2,
         images={"t1": "scalar"},
         transform=("Normalize", {"percentile_low": 0.5, "percentile_high": 99.5, "out_min": 0.0, "out_max": 1.0})),
    dict(name="normalize_random_out_masked", seed=105, shape=(24, 20, 16), batch=3,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Normalize", {"out_min": (-1.0, 0.0), "out_max": (0.5, 1.0), "masking_method": "seg",
                                  "percentile_low": 1.0, "percentile_high": 99.0})),
    dict(name="normalize_explicit_in", seed=106, shape=(16, 14, 12), batch=2,
         images={"t1": "scalar"}, transform=("Normalize", {"in_min": 0.1, "in_max": 0.8})),
]

# ---- remaining Spatial modes (SURVEY §8 f-4): target spaces, anti-aliasing -------------------
_TARGET_AFFINE = [[0.0, -1.3, 0.0, 14.0], [1.1, 0.0, 0.0, -3.0], [0.0, 0.0, 1.6, 2.0], [0.0, 0.0, 0.0, 1.0]]
RESAMPLE_CASES = [
    dict(name="resample_iso2_aniso", seed=111, shape=(20, 18, 14), batch=2, spacing=(0.8, 1.1, 2.0),
         origin=(-7.0, 3.5, 10.0), tilt=0.1, images={"t1": "scalar", "seg": "int16"},
         transform=("Resample", {"target": 2})),
    dict(name="resample_antialias_down", seed=112, shape=(24, 20, 16), batch=2,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Resample", {"target": (2.0, 2.5, 3.0), "antialias": True})),
    dict(name="resample_up_half", seed=113, shape=(12, 10, 8), batch=1,
         images={"t1": "scalar", "seg": "uint8"}, transform=("Resample", {"target": 0.5})),
    dict(name="resample_random_spacing", seed=114, shape=(20, 18, 14), batch=2,
         images={"t1": "scalar"}, transform=("Resample", {"target": (1.5, 2.5), "antialias": True})),
    dict(name="spatial_target_space_affine", seed=115, shape=(18, 16, 14), batch=2, spacing=(1.2, 0.9, 1.5),
         images={"t1": "scalar", "seg": "uint8"},
         transform=("Spatial", {**_AFF, "max_displacement": (1.0, 2.5), "num_control_points": 6,
                                "target": ((14, 20, 12), _TARGET_AFFINE)})),
    # label_interpolation="label" (partial-volume one-hot / argmax, spatial.py:1275-1389)
    dict(name="label_pv_affine", seed=116, shape=(20, 17, 13), batch=2,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Affine", {**_AFF, "label_interpolation": "label", "default_pad_label": 3})),
    dict(name="label_pv_elastic_gated", seed=117, shape=(18, 16, 14), batch=4, spacing=(1.2, 0.9, 1.5),
         images={"seg": "int32"},
         transform=("Spatial", {**_AFF, "max_displacement": (1.0, 2.5), "num_control_points": 6,
                                "label_interpolation": "label", "default_pad_label": 9, "p": 0.6})),
    # axis-aligned down/up-sampling: exact half-voxel positions, i.e. argmax ties everywhere
    dict(name="label_pv_resample_down", seed=118, shape=(20, 18, 14), batch=2,
         images={"t1": "scalar", "seg": "uint8"},
         transform=("Resample", {"target": 2, "label_interpolation": "label"})),
    dict(name="label_pv_resample_up", seed=119, shape=(12, 10, 8), batch=1,
         images={"seg": "int64"}, transform=("Resample", {"target": 0.5, "label_interpolation": "label"})),
    dict(name="label_pv_antialias", seed=120, shape=(24, 20, 16), batch=2,
         images={"t1": "scalar", "seg": "int16"},
         transform=("Resample", {"target": (2.0, 2.5, 3.0), "antialias": True, "label_interpolation": "label"})),
    dict(name="label_pv_onehot_nearest", seed=121, shape=(16, 14, 12), batch=2,
         images={"seg": "uint8"},
         transform=("Affine", {**_AFF, "label_interpolation": "label", "one_hot_label_interpolation": "nearest"})),
    # ---- K1 tile kernels on target grids (see the tile cases of CASES)
    # a permuted, flipped target grid (like _TARGET_AFFINE) of full 16^3 tiles inside the input's field of view
    dict(name="spatial_target_tiles", seed=134, shape=(40, 36, 48), batch=2, spacing=(1.2, 0.9, 1.5),
         images={"t1": "scalar", "seg": "int16"},
         transform=("Spatial", {**_AFF, "max_displacement": (1.0, 2.5), "num_control_points": 6,
                                "target": ((32, 32, 32), [[0.0, -1.3, 0.0, 44.0], [1.1, 0.0, 0.0, -1.0],
                                                          [0.0, 0.0, 1.6, 8.0], [0.0, 0.0, 0.0, 1.0]])})),
    dict(name="resample_down_tiles", seed=135, shape=(48, 48, 64), batch=2, spacing=(0.9, 0.9, 1.0),
         images={"t1": "scalar", "seg": "uint8"}, transform=("Resample", {"target": (1.35, 1.35, 2.0)})),
    dict(name="label_pv_aniso_tiles", seed=136, shape=(40, 36, 48), batch=2, spacing=(0.8, 1.1, 2.0),
         images={"seg": "int16"},
         transform=("Spatial", {**_AFF, "max_displacement": (1.0, 3.0), "num_control_points": 7,
                                "label_interpolation": "label", "default_pad_label": 9})),
]
# the cases above made for the K1 tile kernels (``generate.py tiles`` writes only these)
TILE_CASE_NAMES = ("elastic_aniso_tiles", "elastic_dense_grid_tiles", "affine_half_voxel_fill",
                   "spatial_target_tiles", "resample_down_tiles", "label_pv_aniso_tiles")

# ---- BASELINE.json's own volume size: 256^3 (configs[1] and configs[2], two elements) ----------
# The reference's full outputs are too large to commit (64 MiB per volume): the fixture keeps
# a strided lattice of every output, two dense blocks (a corner with padding/fill, the centre),
# and SHA-256 of the full label maps (bit-exact by construction).
_P_AFF = ("Affine", {"scales": (0.9, 1.1), "degrees": (-10, 10)})
FULL_CASES = [
    dict(name="full256_config2_b2", seed=1234, shape=(256, 256, 256), batch=2,
         images={"t1": "scalar", "seg": "int16"},
         transform=[_P_AFF, ("ElasticDeformation", {})]),
    dict(name="full256_config3_b2", seed=1234, shape=(256, 256, 256), batch=2,
         images={"t1": "scalar", "seg": "int16"},
         transform=[_P_AFF, ("ElasticDeformation", {}), ("BiasField", {}), ("Blur", {"std": (0.0, 2.0)}),
                    ("Noise", {"std": (0.0, 0.25)}), ("Gamma", {"log_gamma": (-0.3, 0.3)})]),
]
FULL_STRIDE, FULL_OFFSET, FULL_BLOCK = 9, (3, 5, 2), 24


def full_views(t):
    """The parts of a (B,C,256,256,256) output the full-size fixture stores."""
    oi, oj, ok = FULL_OFFSET
    n = t.shape[-1]
    c0 = (n - FULL_BLOCK) // 2
    return {
        "lattice": t[..., oi::FULL_STRIDE, oj::FULL_STRIDE, ok::FULL_STRIDE],
        "corner": t[..., :FULL_BLOCK, n - FULL_BLOCK:, :FULL_BLOCK],
        "centre": t[..., c0:c0 + FULL_BLOCK, c0:c0 + FULL_BLOCK, c0:c0 + FULL_BLOCK],
    }


CASES_BY_NAME = {c["name"]: c for c in CASES + NEIGHBOUR_CASES + CALL_CASES + STAT_CASES + RESAMPLE_CASES
                 + FULL_CASES}


# ---- patch path (SURVEY §8 f-2): UniformSampler / Queue / SubjectsLoader -------------

PATCH_CASES = [
    dict(name="queue_shuffled", num_subjects=5, shape=(20, 24, 28), patch_size=(8, 10, 12),
         max_length=12, patches_per_volume=4, batch_size=3, shuffle_subjects=True,
         shuffle_patches=True, seed=11),
    dict(name="queue_in_order", num_subjects=3, shape=(16, 16, 16), patch_size=(16, 8, 8),
         max_length=100, patches_per_volume=5, batch_size=4, shuffle_subjects=False,
         shuffle_patches=False, seed=12),
]
PATCH_CASES_BY_NAME = {c["name"]: c for c in PATCH_CASES}


def patch_subject_data(case, sid):
    """(t1 fp32 (2,I,J,K), seg int16 (1,I,J,K), affine 4x4 float64) of subject ``sid``."""
    import numpy as np
    import torch

    g = torch.Generator().manual_seed(5000 + 17 * sid + case["seed"])
    shape = case["shape"]
    t1 = torch.rand((2, *shape), generator=g)
    seg = (torch.rand((1, *shape), generator=g) * 5).to(torch.int16)
    affine = np.diag([1.0, 1.5, 2.0, 1.0])
    affine[:3, 3] = [10.0 * sid, -5.0, 2.5]
    return t1, seg, affine
