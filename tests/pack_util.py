"""Synthetic variants of the committed part packs for parity tests.

`permuted_pack` re-expresses a part in a coordinate frame whose principal axes are not (1, 2) --
both reference parts have principal axes (1, 2) (bullet_paint_wrapper.py:1294-1300), so the kernels'
generic-axes instantiations (`move_fast_kernel<G, false, ...>` / `paint_kernel<C, ST, false, ...>`) are otherwise
never reached.  The oracle and the engine both consume the transformed pack, so the comparison stays
like against like; derived per-triangle constants (d00 ...) are kept as they are.
"""
import numpy as np

from paintrl_b200.partpack import PartPack

# new[k] = sign[k] * old[src[k]]
FRAMES = {
    # swap x and y: non-principal axis 1, principal axes (0, 2)
    'axes02': ((1, 0, 2), (1.0, 1.0, 1.0)),
    # (y, z, -x): non-principal axis 2 with the tool looking along +z, principal axes (0, 1)
    'axes01': ((1, 2, 0), (1.0, 1.0, -1.0)),
}

_VEC_KEYS = ('planes_n', 'front_pos', 'vertices', 'tri_a', 'tri_v0', 'tri_v1', 'tri_b', 'tri_c', 'tri_n',
             'start_fixed', 'start_anchor', 'start_edge', 'start_all')


def permuted_pack(pack, frame):
    src, sign = FRAMES[frame]
    sign = np.asarray(sign)
    arrays = dict(pack.arrays)
    for key in _VEC_KEYS:
        if key in arrays:
            arrays[key] = np.ascontiguousarray(np.asarray(arrays[key], dtype=np.float64)[..., list(src)] * sign)
    meta = dict(pack.meta)
    old_axes = tuple(pack.axes)
    new_axes = tuple(sorted(src.index(a) for a in old_axes))
    # the transformed frame must keep the ROLE of each principal axis (ranges, silhouette table and the
    # length / width ratio are per axis): old axis0 -> new axis0, old axis1 -> new axis1
    assert new_axes == (src.index(old_axes[0]), src.index(old_axes[1])), 'frame swaps the principal axes'
    assert all(sign[a] > 0 for a in new_axes), 'principal axes must not be mirrored'
    meta['axes'] = list(new_axes)
    meta['non_principal_axis'] = 3 - sum(new_axes)
    meta['source'] = 'synthetic frame %s of %s' % (frame, meta.get('part_name'))
    return PartPack(meta, arrays)


# ------------------------------------------------------------------------------------------ digests
DIGEST_SKIP = ('grid_cells_4', 'grid_cells_10')      # reference-side cross-check tables, not produced by the loader
_PER_TEXEL = ('front_ij', 'front_pos', 'texel_off', 'status_init_rgb', 'status_init_hsi')


def pack_digest(pack):
    """sha256 of every table of a pack, with the front texels brought into (i, j) order first (the reference keeps
    them in `set` iteration order, the loader sorted), plus the scalars of the meta block that the step consumes."""
    import hashlib
    ij = np.asarray(pack.arrays['front_ij'], dtype=np.int64)
    order = np.lexsort((ij[:, 1], ij[:, 0]))
    out = {}
    for key in sorted(pack.arrays):
        if key in DIGEST_SKIP:
            continue
        a = np.asarray(pack.arrays[key])
        if key in _PER_TEXEL:
            a = a[order]
        a = np.ascontiguousarray(a, dtype=np.int64 if a.dtype.kind in 'iu' else np.float64)
        out[key] = '%s:%s' % ('x'.join(str(d) for d in a.shape), hashlib.sha256(a.tobytes()).hexdigest()[:24])
    for key in ('width', 'height', 'axes', 'non_principal_axis', 'front_normal', 'density'):
        out['meta.' + key] = repr(pack.meta[key])
    return out
