"""Generate golden vectors by running the UNMODIFIED reference on CPU.

TEST INFRASTRUCTURE.  Run in the build container only (needs the read-only
reference checkout at /root/reference plus the stub shim in ``_shim/`` for the
I/O-only dependencies that are absent here):

    python tests/golden/generate.py

For every case we record the exact ``params`` dict the reference sampled
(JSON), the seeds needed to regenerate the inputs, and the reference's output
tensors.  Inputs are regenerated from seeds by ``tests/golden_cases.py`` so the
fixtures stay small.  Nothing here is imported by the product.
"""

from __future__ import annotations

import json
import sys
import warnings
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE / "_shim"))
sys.path.insert(1, "/root/reference/src")
sys.path.insert(2, str(HERE.parent))

import torchio as tio  # noqa: E402  (the reference)

from golden_cases import (  # noqa: E402
    CALL_CASES, CASES, CASES_BY_NAME, NEIGHBOUR_CASES, RESAMPLE_CASES, STAT_CASES, TILE_CASE_NAMES, build_inputs)


def _make_transform(spec):
    """Instantiate a reference transform (or Compose) from a case spec."""
    if isinstance(spec, list):
        return tio.Compose([_make_transform(s) for s in spec], copy=False)
    name, kwargs = spec
    return getattr(tio, name)(**kwargs)


def _to_reference_batch(inputs):
    subjects = []
    for sub in inputs["subjects"]:
        kwargs = {}
        for name, (kind, tensor, affine) in sub.items():
            cls = tio.ScalarImage if kind == "scalar" else tio.LabelMap
            kwargs[name] = cls(tensor.clone(), affine=affine.copy())
        subjects.append(tio.Subject(**kwargs))
    return tio.SubjectsBatch.from_subjects(subjects)


def run_case(case):
    inputs = build_inputs(case)
    batch = _to_reference_batch(inputs)
    transform = _make_transform(case["transform"])
    torch.manual_seed(case["seed"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = transform(batch)
    history = [
        {"name": t.name, "params": t.params} for t in out.applied_transforms
    ]
    arrays = {}
    for name, img_batch in out.images.items():
        arrays[f"out_{name}"] = img_batch.data.contiguous().numpy()
        arrays[f"aff_{name}"] = np.stack([a.numpy() for a in img_batch.affines])
    arrays["history"] = np.frombuffer(
        json.dumps(history).encode(), dtype=np.uint8
    )
    return arrays


def _unchanged(path, arrays):
    """True when ``path`` already holds exactly ``arrays`` (the zip container stamps the time of
    writing, so rewriting identical data would still change the file)."""
    if not path.exists():
        return False
    with np.load(path) as z:
        return set(z.files) == set(arrays) and all(
            z[k].dtype == v.dtype and np.array_equal(z[k], v) for k, v in arrays.items())


def main():
    torch.set_num_threads(1)
    out_dir = HERE
    only = sys.argv[1] if len(sys.argv) > 1 else "all"   # "neighbours": leave the hot-path fixtures alone
    selected = {"neighbours": NEIGHBOUR_CASES, "call": CALL_CASES, "stats": STAT_CASES,
                "resample": RESAMPLE_CASES, "tiles": [CASES_BY_NAME[n] for n in TILE_CASE_NAMES]}.get(
        only, CASES + NEIGHBOUR_CASES + CALL_CASES + STAT_CASES + RESAMPLE_CASES)
    for case in selected:
        arrays = run_case(case)
        path = out_dir / f"{case['name']}.npz"
        state = "unchanged" if _unchanged(path, arrays) else "written"
        if state == "written":
            np.savez_compressed(path, **arrays)
        size = path.stat().st_size / 1024
        print(f"{case['name']:40s} {size:8.1f} KiB  {state}")


if __name__ == "__main__":
    main()
