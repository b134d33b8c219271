"""K1 tile kernels against the C oracle (every voxel) on the geometries real data takes: thick
slices, resampling to other grids, permuted and flipped target spaces, elastic grids from coarse
to as dense as the bounds pre-pass accepts, and fill decisions exactly on the mask threshold.

Every case also asserts how many output tiles took the tile walk (the TMA box) rather than the
general column, from the per-tile records of the bounds pre-pass: a change of the heuristics
must not quietly turn these into tests of the general kernel.

Bars: label maps (nearest and partial volume) bit-exact; fp32 with the exact coordinate chain
<= 1e-6 abs, fast coordinates <= 1e-4 abs on data in [-0.25, 0.75]; fill positions identical in
both modes.  The fast coordinates are also held to DESIGN §3: against the real-valued mapping
(float64), no worse than the exact chain plus 1e-6.
"""

from __future__ import annotations

import json
import types
import warnings
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from golden_cases import TILE_CASE_NAMES
from util import load_golden, product_batch, product_replay

pytestmark = pytest.mark.gpu

TILED_LABELS = (torch.uint8, torch.int16, torch.int32)
WALK_FLOOR = 0.3  # fraction of tiles that must take the tile walk where the geometry is made to


# ---- the kernel call, keeping the bounds records ----------------------------------------------


def k1(src, mat, cp, flags, sp_in, sp_out, *, affine_first, mode, fill, out_shape=None, box_hint=0,
       exact):
    """``tio_resample`` called as ``ops.resample`` calls it, except that the workspace is zeroed
    first and kept.  Returns (output, records): records is (B, tiles_i, tiles_j, tiles_k, 4) int32
    (origin of the staged box, flags word) or None when no tile path was asked for.  A launch the
    tile path refuses leaves the zeroed records, i.e. no tile walks."""
    from torchio_b200 import _native, ops

    src = src.contiguous()
    b, c, i, j, k = src.shape
    oi, oj, ok = (i, j, k) if out_shape is None else out_shape
    dst = torch.empty((b, c, oi, oj, ok), dtype=src.dtype, device=src.device)
    ni = nj = nk = 0
    if cp is not None:
        ni, nj, nk = cp.shape[1:4]
    spi = np.asarray(sp_in, dtype=np.float32)
    spo = np.asarray(sp_out, dtype=np.float32)
    workspace, ws_bytes = None, 0
    if box_hint >= 0:
        ws_bytes = _native.lib().tio_resample_workspace_bytes(b, oi, oj, ok)
        workspace = torch.zeros(ws_bytes, dtype=torch.uint8, device=src.device)
    ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    with torch.cuda.device(src.device):
        _native.call(
            "tio_resample", ptr(src), ptr(dst), ops.DTYPE_CODES[src.dtype], b, c, i, j, k, oi, oj, ok,
            ptr(mat), ptr(cp), ptr(flags), ni, nj, nk, spi.ctypes.data, spo.ctypes.data,
            int(bool(affine_first)), int(mode) | (ops.EXACT_COORDS if exact else 0), ptr(fill),
            int(box_hint), ptr(workspace), ws_bytes, torch.cuda.current_stream(src.device).cuda_stream)
    records = None
    if workspace is not None:
        tiles = [(n + 15) // 16 for n in (oi, oj, ok)]
        records = workspace.view(torch.int32).reshape(b, *tiles, 4).cpu()
    return dst, records


def walked(records, *, dtype, mode, exact, has_fill):
    """Boolean (B, tiles...) of the tiles that walked the staged box, and the mask of the tiles
    that were not pass-through elements (code 3).  Flags word (resample_tile.cuh, tile_bounds_kernel):
    bits 0-7 fit code (1 = fits the box), bit 8 every tap in bounds, bit 11 full 16^3 tile.
      fast kernel (fp32 linear, fast coordinates): code 1 and a full tile (resample_fast.cu);
      tile kernel (exact fp32, nearest, partial volume): code 1, ragged tiles included, except
      nearest with a fill value on a tile touching the border (resample_tile.cu)."""
    from torchio_b200 import ops

    w = records[..., 3]
    code = w & 255
    live = code != 3
    if dtype == torch.float32 and mode == ops.LINEAR and not exact:
        walk = (w & (255 | 2048)) == (1 | 2048)
    else:
        walk = code == 1
        if mode == ops.NEAREST and has_fill:
            walk &= (w & 256) != 0
    return walk & live, live


def walked_fraction(records, **kw):
    walk, live = walked(records, **kw)
    return float(walk.sum()) / max(int(live.sum()), 1)


def check_floor(frac, *, walk, mode, has_fill, what):
    """walk: at least WALK_FLOOR of the tiles took the tile walk; no walk: none did.  Nearest with a
    fill value walks only the tiles whose every tap is inside the volume (border tiles need the
    per-voxel mask of the general column), so its share is a property of the geometry: reported only."""
    from torchio_b200 import ops

    if not walk:
        assert frac == 0.0, (what, frac)
    elif not (mode == ops.NEAREST and has_fill):
        assert frac >= WALK_FLOOR, (what, frac)


# ---- geometry -----------------------------------------------------------------------------------


def _rotation(angles):
    cx, sx, cy, sy, cz, sz = (f(a) for a in angles for f in (np.cos, np.sin))
    rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return rz @ ry @ rx


def _space(shape, spacing, origin=(0.0, 0.0, 0.0)):
    a = np.diag([*spacing, 1.0])
    a[:3, 3] = origin
    return a


def geometry(case, rng):
    """(out_shape, a_in, a_out, worlds, cps) of a geometry case; worlds are the world transforms
    T of the elements (the kernel's matrix is inv(A_in) inv(T) A_out), cps (B, ni, nj, nk, 3) mm."""
    from oracle import torch_port

    shape, b = case["shape"], case["batch"]
    sp_in = np.asarray(case["sp_in"], dtype=np.float64)
    a_in = _space(shape, sp_in, (3.0, -2.0, 5.0))
    extent = np.asarray(shape) * sp_in
    grid = case["grid"]
    if grid == "perm":  # rows swapped, negative entries (a target space like _TARGET_AFFINE)
        out_shape = (32, 32, 112)
        a_out = np.array([[0.0, -1.3, 0.0, 3.0 + extent[0] - 2.0], [1.1, 0.0, 0.0, -1.0],
                          [0.0, 0.0, 1.6, 6.0], [0.0, 0.0, 0.0, 1.0]])
    else:
        sp_out = np.asarray(case.get("sp_out") or sp_in * case.get("zoom", 1.0), dtype=np.float64)
        out_shape = tuple(int(round(n)) for n in extent / sp_out)
        # voxel centres of the output grid inside the input's field of view
        a_out = _space(out_shape, sp_out, a_in[:3, 3] + (sp_out - sp_in) / 2)
    centre = a_in[:3, :3] @ ((np.asarray(shape) - 1) / 2) + a_in[:3, 3]
    worlds = []
    for _ in range(b):
        t = np.eye(4)
        if case.get("half_voxel"):
            t[:3, :3] = _rotation((0.0, 0.0, case.get("tiny_angle", 0.0)))
            t[:3, 3] = (0.5, -1.5, 2.5)
        else:
            r = _rotation(rng.uniform(-case["rot"], case["rot"], 3))
            t[:3, :3] = r
            t[:3, 3] = centre - r @ centre + rng.uniform(-case["shift"], case["shift"], 3)
        worlds.append(t)
    cps = None
    if case.get("cp"):
        n_cp, mm = case["cp"]
        cps = np.stack([rng.uniform(-1, 1, (*n_cp, 3)) * np.asarray(mm) for _ in range(b)]).astype(np.float32)
    mats = np.stack([torch_port.output_to_input_matrix(a_in, a_out, t).numpy()[:3].reshape(12) for t in worlds])
    return out_shape, a_in, a_out, worlds, cps, mats


def grid64(mat, cp, sp_in, sp_out, out_shape, affine_first):
    """Input-voxel coordinates of every output voxel in float64: the real-valued mapping of the
    kernel's fp32 tables (matrix, control grid, spacings)."""
    from oracle import torch_port

    coords = torch_port.voxel_coordinates(out_shape).double()
    m = torch.as_tensor(np.asarray(mat, dtype=np.float64).reshape(3, 4))
    aff = lambda p: p @ m[:, :3].T + m[:, 3]  # noqa: E731
    if cp is None:
        return aff(coords)
    field = torch.as_tensor(cp, dtype=torch.float64).permute(3, 0, 1, 2)[None]
    disp = F.interpolate(field, size=list(out_shape), mode="trilinear", align_corners=True)[0].permute(1, 2, 3, 0)
    if affine_first:
        return aff(coords) + disp / torch.as_tensor(np.float32(sp_in), dtype=torch.float64)
    return aff(coords + disp / torch.as_tensor(np.float32(sp_out), dtype=torch.float64))


def sample64(data, vox):
    """Trilinear sampling of (C,I,J,K) data at float64 voxel coordinates (zeros outside)."""
    in_shape = data.shape[1:]
    sizes = torch.tensor([max(n - 1, 1) for n in in_shape], dtype=torch.float64)
    g = (2.0 * vox / sizes - 1.0).permute(2, 1, 0, 3)[None]  # (1, K, J, I, 3)
    x = data.double().permute(0, 3, 2, 1)[None]
    return F.grid_sample(x, g, mode="bilinear", padding_mode="zeros", align_corners=True)[0].permute(0, 3, 2, 1)


# ---- the geometry matrix -------------------------------------------------------------------------
# walk: True = at least WALK_FLOOR of the tiles take the tile walk at the box the transforms pick
# (spatial._box_hint), False = none may (the geometry is made to fall back).

_ANISO = (0.8, 1.1, 2.0)
GEOMETRIES = [
    dict(name="unit_same", shape=(64, 48, 80), batch=3, channels=2, sp_in=(1, 1, 1), grid="same",
         rot=0.2, shift=4.0, walk=True),
    dict(name="unit_same_fill_c3", shape=(64, 48, 80), batch=3, channels=3, sp_in=(1, 1, 1), grid="same",
         rot=0.15, shift=8.0, fill=(-1.0, 0.5, 0.25), walk=True),
    dict(name="aniso_same_cp7", shape=(64, 48, 80), batch=3, channels=2, sp_in=_ANISO, grid="same",
         rot=0.15, shift=4.0, cp=((7, 7, 7), 6.0), fill=(-1.0, 0.5), walk=True),
    dict(name="thick_to_iso15_cp7", shape=(96, 80, 48), batch=3, channels=2, sp_in=(0.9, 0.9, 3.0),
         sp_out=(1.5, 1.5, 1.5), grid="spacing", rot=0.03, shift=3.0, cp=((7, 7, 7), 1.0), fill=(0.0, -0.5),
         walk=True),
    dict(name="aniso_up2_cells", shape=(32, 24, 48), batch=2, channels=2, sp_in=_ANISO, zoom=0.5, grid="zoom",
         rot=0.1, shift=2.0, cp=((13, 10, 19), tuple(0.5 * 5.2 * s / 2 for s in _ANISO)), walk=True),
    dict(name="unit_down14", shape=(96, 80, 112), batch=3, channels=2, sp_in=(1, 1, 1), zoom=1.4, grid="zoom",
         rot=0.05, shift=3.0, fill=(-1.0, 0.5), walk=True),
    dict(name="thick_down2_rotated", shape=(64, 48, 80), batch=3, channels=2, sp_in=(0.9, 0.9, 3.0), zoom=2.0,
         grid="zoom", rot=0.2, shift=3.0, walk=False),
    dict(name="aniso_perm_flip", shape=(48, 40, 96), batch=3, channels=2, sp_in=_ANISO, grid="perm",
         rot=0.02, shift=2.0, cp=((7, 7, 7), 0.5), fill=(-1.0, 0.5), walk=True),
    # cells of ~5.2-6.5 voxels at +- half a cell: the densest grid every tile of the pre-pass accepts
    dict(name="unit_cells_half", shape=(64, 48, 80), batch=3, channels=2, sp_in=(1, 1, 1), grid="same",
         rot=0.05, shift=2.0, cp=((13, 9, 14), 2.6), fill=(-1.0, 0.5), walk=True),
    # cells of ~3.5 voxels: more than two cell crossings per tile axis, the pre-pass gives up
    dict(name="aniso_dense_grid", shape=(64, 48, 80), batch=3, channels=2, sp_in=_ANISO, grid="same",
         rot=0.05, shift=2.0, cp=((19, 14, 23), 1.0), fill=(-1.0, 0.5), walk=False),
    # half-voxel translations: masks of exactly 0.5 (decided by the last bit of the fp32 chain), then
    # a 1e-7 rad rotation that moves them into the band the fast kernel recomputes exactly
    dict(name="half_voxel", shape=(40, 36, 48), batch=1, channels=2, sp_in=(1, 1, 1), grid="same",
         half_voxel=True, fill=(-1.0, 0.5), walk=True),
    dict(name="half_voxel_tiny_rotation", shape=(40, 36, 48), batch=1, channels=2, sp_in=(1, 1, 1), grid="same",
         half_voxel=True, tiny_angle=1e-7, fill=(-1.0, 0.5), walk=True),
]


def _oracle(data, mat, cp, flags, sp_in, sp_out, out_shape, affine_first, mode, fill):
    from oracle import c_port

    b, c = data.shape[:2]
    want = torch.empty((b, c, *out_shape), dtype=data.dtype)
    ni, nj, nk = (0, 0, 0) if cp is None else cp.shape[1:4]
    p = c_port._p
    # (held in locals: a temporary tensor would be freed, and its memory reused, before the call)
    spi, spo = torch.as_tensor(np.float32(sp_in)), torch.as_tensor(np.float32(sp_out))
    rc = c_port.lib().orc_resample(
        p(data), p(want), c_port._DTYPES[data.dtype], b, c, *data.shape[2:], *out_shape, p(mat), p(cp), p(flags),
        ni, nj, nk, p(spi), p(spo), int(affine_first), mode, p(fill))
    assert rc == 0
    return want


def _blocky_labels(b, shape):
    i, j, k = (torch.arange(n) for n in shape)
    lab = ((i[:, None, None] // 5) * 3 + (j[None, :, None] // 7) * 5 + (k[None, None, :] // 6)) % 6
    return torch.stack([(lab * (2 * e + 1) + e) % 6 for e in range(b)])[:, None].contiguous()


@pytest.mark.parametrize("case", GEOMETRIES, ids=[g["name"] for g in GEOMETRIES])
def test_tile_kernels_match_oracle_on_every_voxel(case):
    from oracle import torch_port
    from torchio_b200 import ops
    from torchio_b200.transforms import spatial

    rng = np.random.default_rng(zlib.crc32(case["name"].encode()))
    out_shape, a_in, a_out, worlds, cps, mats = geometry(case, rng)
    b, c, shape = case["batch"], case["channels"], case["shape"]
    sp_in, sp_out = torch_port.spacing_of(a_in), torch_port.spacing_of(a_out)
    g = torch.Generator().manual_seed(7)
    data = torch.rand((b, c, *shape), generator=g) - 0.25
    fill = None if case.get("fill") is None else torch.tensor(case["fill"], dtype=torch.float32)
    hint = spatial._box_hint(types.SimpleNamespace(mat=mats, cp=cps), sp_in, sp_out, out_shape)
    dev = torch.device("cuda")
    mat_d = torch.as_tensor(mats).to(dev)
    cp_d = None if cps is None else torch.as_tensor(cps).to(dev)
    fill_d = None if fill is None else fill.to(dev)
    data_d = data.to(dev)
    variants = [(True, None)]
    if cps is not None:  # both composition orders, the last element gated: a bit copy on the same grid,
        # the identity resampling onto another one (the transforms pass nothing through to a target)
        gated = 1 if tuple(out_shape) == tuple(shape) else 0
        variants = [(True, np.full(b, 2, np.uint8)), (False, np.array([2] * (b - 1) + [gated], np.uint8))]
    lines = [f"{case['name']}: in {shape} -> out {out_shape}, sp {tuple(round(x, 4) for x in sp_in)} -> "
             f"{tuple(round(x, 4) for x in sp_out)}, auto box {hint}"]
    for affine_first, flags in variants:
        fl_t = None if flags is None else torch.as_tensor(flags)
        fl_d = None if fl_t is None else fl_t.to(dev)
        cp_t = None if cps is None else torch.as_tensor(cps)
        tag = f"affine_first={affine_first}"
        # ---- fp32 trilinear -----------------------------------------------------------------------
        want = _oracle(data, torch.as_tensor(mats), cp_t, fl_t, sp_in, sp_out, out_shape, affine_first,
                       ops.LINEAR, fill)
        got = {}
        for exact in (True, False):
            for box in (hint, 0, 20, 24, 32):
                out, rec = k1(data_d, mat_d, cp_d, fl_d, sp_in, sp_out, affine_first=affine_first, mode=ops.LINEAR,
                              fill=fill_d, out_shape=out_shape, box_hint=box, exact=exact)
                out = out.cpu()
                frac = walked_fraction(rec, dtype=torch.float32, mode=ops.LINEAR, exact=exact,
                                       has_fill=fill is not None)
                err = float((out - want).abs().max())
                bar = 1e-6 if exact else 1e-4
                lines.append(f"  {tag} fp32 {'exact' if exact else 'fast '} box {box:2d}: walked {frac:.2f}, "
                             f"max |err| vs oracle {err:.2e}")
                assert err <= bar, (case["name"], tag, exact, box, err)
                if fill is not None:
                    for ch in range(c):
                        assert torch.equal(out[:, ch] == fill[ch], want[:, ch] == fill[ch]), (tag, exact, box, ch)
                if flags is not None and flags[-1] == 1:
                    assert torch.equal(out[-1], data[-1])
                if box == hint:
                    check_floor(frac, walk=case["walk"], mode=ops.LINEAR, has_fill=fill is not None,
                                what=(case["name"], tag, exact))
                    got[exact] = out
        # the fast form against the real-valued mapping: no worse than the exact chain (DESIGN §3)
        errs = {True: 0.0, False: 0.0}
        for e in range(b):
            if flags is not None and flags[e] & 1:
                continue
            vox = grid64(mats[e], None if cps is None or not flags[e] & 2 else cps[e], sp_in, sp_out, out_shape,
                         affine_first)
            inside = torch.ones(out_shape, dtype=torch.bool)
            for ax, n in enumerate(shape):
                inside &= (vox[..., ax] >= 1e-3) & (vox[..., ax] <= n - 1 - 1e-3)
            ref = sample64(data[e], vox)
            for exact in (True, False):
                d = (got[exact][e].double() - ref).abs()[:, inside]
                errs[exact] = max(errs[exact], float(d.max()) if d.numel() else 0.0)
        lines.append(f"  {tag} fp32 vs float64 mapping: exact {errs[True]:.2e}, fast {errs[False]:.2e}")
        assert errs[False] <= errs[True] + 1e-6, (case["name"], tag, errs)
        # ---- label maps, nearest: bit-exact with the oracle for every tiled dtype ------------------
        lab = torch.randint(0, 100, (b, 1, *shape), generator=g, dtype=torch.int32)
        lab_fill = None if fill is None else torch.tensor([7.0])
        want_l = _oracle(lab, torch.as_tensor(mats), cp_t, fl_t, sp_in, sp_out, out_shape, affine_first,
                         ops.NEAREST, lab_fill)
        for dtype in TILED_LABELS:
            out, rec = k1(lab.to(dtype).to(dev), mat_d, cp_d, fl_d, sp_in, sp_out, affine_first=affine_first,
                          mode=ops.NEAREST, fill=None if lab_fill is None else lab_fill.to(dev), out_shape=out_shape,
                          box_hint=hint, exact=True)
            frac = walked_fraction(rec, dtype=dtype, mode=ops.NEAREST, exact=True, has_fill=lab_fill is not None)
            mism = int((out.cpu().to(torch.int32) != want_l).sum())
            lines.append(f"  {tag} nearest {str(dtype)[6:]:5s}: walked {frac:.2f}, mismatches {mism}")
            assert mism == 0, (case["name"], tag, dtype, mism)
            check_floor(frac, walk=case["walk"], mode=ops.NEAREST, has_fill=lab_fill is not None,
                        what=(case["name"], tag, dtype))
        # ---- label maps, partial volume: tile == general, == the one-hot / grid_sample / argmax port --
        blocky = _blocky_labels(b, shape)
        pad = torch.tensor([9.0])
        general = None
        for dtype in TILED_LABELS:
            src = blocky.to(dtype).to(dev)
            kw = dict(affine_first=affine_first, mode=ops.LABEL_PV, fill=pad.to(dev), out_shape=out_shape, exact=True)
            tiled, rec = k1(src, mat_d, cp_d, fl_d, sp_in, sp_out, box_hint=hint, **kw)
            ref, _ = k1(src, mat_d, cp_d, fl_d, sp_in, sp_out, box_hint=-1, **kw)
            frac = walked_fraction(rec, dtype=dtype, mode=ops.LABEL_PV, exact=True, has_fill=True)
            mism = int((tiled != ref).sum())
            lines.append(f"  {tag} label_pv {str(dtype)[6:]:5s}: walked {frac:.2f}, tile vs general mismatches {mism}")
            assert mism == 0, (case["name"], tag, dtype, mism)
            check_floor(frac, walk=case["walk"], mode=ops.LABEL_PV, has_fill=True, what=(case["name"], tag, dtype))
            general = ref.cpu().to(torch.int32) if general is None else general
            assert torch.equal(ref.cpu().to(torch.int32), general)
        for e in range(b):
            if flags is not None and flags[e] & 1:
                assert torch.equal(general[e], blocky[e].to(torch.int32))
                continue
            cp_e = None if cps is None or not flags[e] & 2 else cps[e]
            vox = torch_port.sampling_grid(shape, a_in, out_shape, a_out, worlds[e], cp_e, affine_first)
            want_pv = torch_port.label_partial_volume(blocky[e:e + 1], vox, shape, a_in, a_out, False, "linear", 9.0)
            mism = int((general[e:e + 1] != want_pv.to(torch.int32)).sum())
            assert mism == 0, (case["name"], tag, e, mism)
    print("\n".join(lines))


# ---- golden fixtures made for the tile kernels: they must keep reaching them ---------------------


def _recording_resample(log):
    """Drop-in for ops.resample that runs ``k1`` and logs the walked fraction of every launch."""
    from torchio_b200 import ops

    def resample(src, mat, cp, flags, spacing_in, spacing_out, *, affine_first, mode, fill, out_shape=None,
                 box_hint=0, exact_coords=None):
        exact = ops.exact_coords_default() if exact_coords is None else exact_coords
        out, rec = k1(src, mat, cp, flags, spacing_in, spacing_out, affine_first=affine_first, mode=mode,
                      fill=fill, out_shape=out_shape, box_hint=box_hint, exact=exact)
        if rec is not None:
            frac = walked_fraction(rec, dtype=src.dtype, mode=mode, exact=exact, has_fill=fill is not None)
            log.append((str(src.dtype)[6:], mode, fill is not None, frac))
        return out

    return resample


@pytest.mark.parametrize("name", TILE_CASE_NAMES)
def test_tile_fixtures_reach_the_tile_walk(name, coords, monkeypatch):
    """The recorded params of each tile fixture, replayed through the transforms (tables.spatial_tables
    and spatial._box_hint as the transforms build them): every K1 launch walks at least WALK_FLOOR
    of its tiles, and the result still equals the reference."""
    from torchio_b200 import ops

    _, images, history, expected, _ = load_golden(name)
    log = []
    monkeypatch.setattr(ops, "resample", _recording_resample(log))
    out = product_replay(product_batch(images, device="cuda"), history)
    print(f"{name} ({coords}): " + ", ".join(f"{d} mode {m} fill {h} walked {f:.2f}" for d, m, h, f in log))
    assert log
    for dtype, mode, has_fill, frac in log:
        check_floor(frac, walk=True, mode=mode, has_fill=has_fill, what=(name, dtype, mode))
    for n, exp in expected.items():
        got = out.images[n].data.cpu()
        if images[n]["kind"] == "label":
            assert torch.equal(got, exp), (n, int((got != exp).sum()))
        else:
            assert float((got - exp).abs().max()) <= 1e-4, n


# ---- a clinical shape: thick axial slices ------------------------------------------------------------


def test_clinical_thick_slices_match_oracle(coords, monkeypatch):
    """(2, 1, 256, 256, 48) at 0.9 x 0.9 x 3 mm through a sampled Affine then a default
    ElasticDeformation: fp32 and int16 labels against the C oracle on every voxel."""
    import torchio_b200 as tio
    from oracle import c_port
    from torchio_b200 import ops

    shape, sp = (256, 256, 48), (0.9, 0.9, 3.0)
    g = torch.Generator().manual_seed(21)
    affine = np.diag([*sp, 1.0])
    images = {
        "t1": {"kind": "scalar", "data": torch.rand((2, 1, *shape), generator=g) - 0.25, "affines": [affine] * 2},
        "seg": {"kind": "label", "data": _blocky_labels(2, shape).to(torch.int16), "affines": [affine] * 2},
    }
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pipe = tio.Compose([tio.Affine(scales=(0.9, 1.1), degrees=(-10, 10)), tio.ElasticDeformation()])
    log = []
    monkeypatch.setattr(ops, "resample", _recording_resample(log))
    torch.manual_seed(3)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = pipe(product_batch(images, device="cuda"))
    history = json.loads(json.dumps([{"name": t.name, "params": t.params} for t in out.applied_transforms]))
    want = c_port.replay({n: dict(v, data=v["data"].clone()) for n, v in images.items()}, history)
    print(f"clinical ({coords}): " + ", ".join(f"{d} mode {m} fill {h} walked {f:.2f}" for d, m, h, f in log))
    assert log
    for dtype, mode, has_fill, frac in log:
        check_floor(frac, walk=True, mode=mode, has_fill=has_fill, what=("clinical", dtype, mode))
    got_l = out.images["seg"].data.cpu()
    assert torch.equal(got_l, want["seg"]["data"]), int((got_l != want["seg"]["data"]).sum())
    err = float((out.images["t1"].data.cpu() - want["t1"]["data"]).abs().max())
    print(f"clinical ({coords}): fp32 max |err| vs oracle {err:.2e}")
    assert err <= (1e-6 if coords == "exact" else 1e-4), err
