"""The part loader (paintrl_b200/loader.py) against the reference's own load-time results.

* `bulge` is the repository's synthetic part (tests/data/make_synthetic_part.py); tests/golden/bulge_128x128.npz is the
  pack the REFERENCE made of it (oracle/make_golden.py pack100: PaintRL's own `load_part` under shims S1-S5).  The loader
  must reproduce every table bit for bit -- with the C oracle's rasteriser here, with the GPU rasteriser under `-m gpu`.
* The reference's parts (door_test, square, door_rr, test: committed packs; door_lf, door_lr, door_rf, roof, bonnet,
  door_rr_big: digests of reference-minted packs, tests/golden/pack_digests.json) are checked when PAINTRL_REFERENCE
  names a checkout of the reference, whose meshes this repository does not carry.
"""
import json
import os

import numpy as np
import pytest

from pack_util import DIGEST_SKIP, pack_digest
from paintrl_b200 import loader
from paintrl_b200.partpack import PART_DICT, PartPack

HERE = os.path.dirname(os.path.abspath(__file__))
BULGE_URDF = os.path.join(HERE, 'data', 'urdf', 'painting', 'bulge.urdf')
BULGE_GOLDEN = os.path.join(HERE, 'golden', 'bulge_128x128.npz')
REF_PARTS = os.path.join(os.environ.get('PAINTRL_REFERENCE', ''), 'PaintRLEnv', 'urdf', 'painting')
needs_reference = pytest.mark.skipif(not os.environ.get('PAINTRL_REFERENCE') or not os.path.isfile(os.path.join(REF_PARTS, 'door_test.urdf')),
                                     reason='PAINTRL_REFERENCE does not name a checkout of the reference with its part meshes')


def oracle_rasterizer(*args):
    from oracle import oracle          # the checker's rasteriser stands in for the GPU one on CPU-only machines
    return oracle.rasterize(*args)


def assert_same_tables(made, ref):
    made = made.reordered_like(ref)
    for key, want in ref.arrays.items():
        if key in DIGEST_SKIP:
            continue
        got = made.arrays[key]
        assert got.shape == want.shape, key
        assert np.array_equal(got, want), key
    for key in ('width', 'height', 'axes', 'non_principal_axis', 'front_normal', 'density', 'max_points'):
        assert made.meta[key] == ref.meta[key], key


def test_synthetic_part_matches_the_reference_pack():
    made = loader.load_part(BULGE_URDF, max_points=5200, part_no=100, rasterizer=oracle_rasterizer)
    assert_same_tables(made, PartPack.load(BULGE_GOLDEN))
    stats = made.meta['loader_stats']
    # the part was built so that every branch of the load has work
    assert stats['sparse_grid_rows'] > 0 and stats['hull_corrected_normals'] > 0 and stats['smoothed_normals'] > 0
    assert {m: made.starts[m].shape[0] for m in made.starts} == {'fixed': 1, 'anchor': 4, 'edge': 184, 'all': 1280}


def test_loader_output_is_a_usable_pack():
    made = loader.load_part(BULGE_URDF, max_points=5200, part_no=100, rasterizer=oracle_rasterizer)
    assert made.status_init('RGB') == 191 and made.status_init('HSI') == 255
    assert np.array_equal(made.texel_offsets(), made.arrays['texel_off'])
    ij = made.front_ij.astype(np.int64)
    assert np.all(np.diff(ij[:, 0] * made.height + ij[:, 1]) > 0), 'texels sorted by (i, j), no duplicates'
    cpack, keep = made.to_c('all', 'RGB')
    assert cpack.n_texels == made.n_texels and cpack.n_starts == 1280


def test_label_texture_keeps_the_reference_quirks():
    # 3 x 2 texture; texel offset = (i + j * W) * 3, the last pixel's is clamped to len - 4
    w, h = 3, 2
    pixels = np.arange(1, w * h * 3 + 1, dtype=np.uint8)
    pixels[0] = 0          # pixel (0, 0): first byte already equals the irrelevant label's -> left alone
    pixels[3] = 191        # pixel (1, 0): first byte already equals the front label's -> left alone
    front = np.array([[1, 0], [2, 0]], dtype=np.int32)
    back = np.array([[0, 1]], dtype=np.int32)
    tex = loader.label_texture(pixels, w, h, front, back, 'RGB')
    assert list(tex[0:3]) == [0, 2, 3]                 # untouched: is_changed() saw 0 == 0
    assert list(tex[3:6]) == [191, 5, 6]               # untouched: 191 == 191
    assert list(tex[6:9]) == [191, 191, 191]           # front
    assert list(tex[9:12]) == [0, 255, 0]              # back
    # (1, 1) irrelevant; (2, 1) is the last pixel: its label lands on bytes len-4 .. len-2, and since (1, 1) has
    # already zeroed byte len-4, is_changed() holds and it is skipped
    assert list(tex[12:15]) == [0, 0, 0] and list(tex[15:18]) == [16, 17, 18]
    assert loader.label_texture(pixels, w, h, front, back, 'HSI')[6] == 255


def test_obj_and_urdf_parsing(tmp_path):
    obj, texture = loader.related_files(BULGE_URDF)
    assert os.path.basename(obj) == 'bulge.obj' and os.path.basename(texture) == 'bulge.png'
    assert os.path.basename(loader.collision_mesh_file(BULGE_URDF)) == 'bulge.obj'
    p = tmp_path / 'm.obj'
    p.write_text('v 0 0 0\nv 1 0 0\nv 0 1 0\nv 0 0 1\nvn 0 0 1\nvt 0.25 0.75\nvt 0 0\nvt 1 1\n\nf 1/1 2/2 3/3\nf 1/1 2/2 3/3 4/1\n')
    v, vt, fv, ft = loader.read_obj(str(p))
    assert len(v) == 4 and vt[0] == [0.25, 0.25]       # v flipped (bullet_paint_wrapper.py:1199)
    assert fv.tolist() == [[0, 1, 2]] and ft.tolist() == [[0, 1, 2]]      # the quad is ignored (:1238)
    bare = tmp_path / 'bare.urdf'
    bare.write_text('<robot name="x"><link name="l"/></robot>')
    assert loader.related_files(str(bare)) == (None, None)


def test_silhouette_walk_on_a_cube():
    # a unit cube's planes and four vertices: the sorted walk of Part._set_grid_dict consumes one vertex per grid row
    # (each band up to the first vertex at or above its upper edge holds at most one: the sparse branch), marches from it
    # to the first 1 mm step that leaves the hull on either side, and reports (0, 0) once the vertices are used up
    n = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], dtype=np.float64)
    off = np.array([1, 0, 1, 0, 1, 0], dtype=np.float64)
    verts = np.array([[0.5, 0.3, 0.1], [0.5, 0.7, 0.1], [0.5, 0.4, 0.95], [0.5, 0.6, 0.95]])
    s = loader.Silhouette(verts, (1, 2), 0, [[0.0, 1.0], [0.0, 1.0]], n, off)
    assert s.sparse_rows == 4 and s.scans == 8
    for row in range(4):
        assert -2e-3 < s.lo[row] < 0.0 and 1.0 < s.hi[row] < 1.0 + 2e-3
    assert not s.lo[4:].any() and not s.hi[4:].any()
    # the sparse branch moved the walk's bound vertex (bullet_paint_wrapper.py:944-947), the other rows are untouched
    assert not np.array_equal(s.data, verts) and np.array_equal(s.data[1:], verts[1:])


@needs_reference
@pytest.mark.parametrize('part_no', [0, 1, 5, 9])
def test_reference_parts_match_the_committed_packs(part_no):
    made = loader.load_part(os.path.join(REF_PARTS, PART_DICT[part_no][0]), rasterizer=oracle_rasterizer)
    assert_same_tables(made, PartPack.for_part(part_no))


@needs_reference
@pytest.mark.parametrize('part_no', [2, 3, 4, 6, 7, 8])
def test_unpacked_reference_parts_match_the_reference_digests(part_no):
    with open(os.path.join(HERE, 'golden', 'pack_digests.json')) as f:
        want = json.load(f).get(os.path.splitext(PART_DICT[part_no][0])[0])
    if want is None:
        pytest.skip('no reference digest for this part (oracle/make_golden.py digests)')
    made = loader.load_part(os.path.join(REF_PARTS, PART_DICT[part_no][0]), rasterizer=oracle_rasterizer)
    got = pack_digest(made)
    assert {k: got[k] for k in want} == want


@pytest.mark.gpu
def test_gpu_rasteriser_path_matches_the_reference_pack(cuda_device):
    made = loader.load_part(BULGE_URDF, max_points=5200, part_no=100)
    assert_same_tables(made, PartPack.load(BULGE_GOLDEN))
    stats = made.meta['loader_stats']
    assert stats['gpu_stages'] and stats['silhouette_scans'] == 200 and stats['silhouette_batches'] > 1


@pytest.mark.gpu
def test_gpu_silhouette_march_matches_the_host_march(cuda_device):
    """`paintrl_silhouette_march` against `march_host` on the synthetic part's hull: scans from random points inside and
    outside the part, both directions, including scans that never leave (found = 0) because the range is cut short."""
    v = loader.read_obj(loader.collision_mesh_file(BULGE_URDF))[0]
    n, off = loader.hull_half_spaces(loader.to_world(v, list(loader.BASE_POSITION)))
    rng = np.random.default_rng(5)
    lo, hi = np.array([-0.45, -0.7, 0.2]), np.array([-0.25, 0.3, 1.3])
    pts = rng.uniform(lo, hi, size=(300, 3))
    is_min = rng.integers(0, 2, size=300).astype(bool)
    for steps_range in (800, 37):
        want_b, want_f = loader.march_host(n, off, pts, is_min, 1, 0, steps_range)
        got_b, got_f = loader.march_gpu(n, off, pts, is_min, 1, 0, steps_range)
        assert np.array_equal(want_f, got_f)
        assert np.array_equal(want_b[want_f], got_b[got_f])
        assert want_f.any() and (steps_range == 800 or not want_f.all())


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['rgb_section', 'hsi_grid_continuous', 'normal_paint'])
def test_loaded_pack_steps_like_the_oracle(case, cuda_device):
    """A pack made by the loader (GPU rasteriser) drives the engine: batches against the C oracle on the same pack."""
    from test_gpu_oracle_batch import BASE, _run_case
    pack = loader.load_part(BULGE_URDF, max_points=5200, part_no=100)
    extra, kw = {
        'rgb_section': (dict(BASE, START_POINT_MODE='all', EPISODE_MAX_LENGTH=40), {}),
        'hsi_grid_continuous': (dict(BASE, START_POINT_MODE='edge', COLOR_MODE='HSI', OVERLAP_PENALTY=True, TURNING_PENALTY=True,
                                     TERMINATION_MODE='hybrid'),
                                dict(action_mode='continuous', action_shape=2, obs_mode='grid', obs_grad=4)),
        'normal_paint': (dict(BASE, START_POINT_MODE='anchor', EPISODE_MAX_LENGTH=30), dict(paint_method='normal')),
    }[case]
    episodes = _run_case(extra, kw, 48, 45, cuda_device, pack=pack)
    assert episodes > 0


def test_load_part_error_paths(tmp_path):
    # a URDF whose mesh has no MTL / texture: the reference's own message (bullet_paint_wrapper.py:1331)
    (tmp_path / 'raw.obj').write_text('v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n')
    urdf = tmp_path / 'raw.urdf'
    urdf.write_text('<robot name="r"><link name="l"><visual><geometry><mesh filename="raw.obj"/></geometry></visual></link></robot>')
    with pytest.raises(FileNotFoundError, match='processed by Blender'):
        loader.load_part(str(urdf), max_points=1, part_no=0, rasterizer=oracle_rasterizer)
    # a part that is not in Part_Dict needs its max-points value
    with pytest.raises(ValueError, match='max_points'):
        loader.load_part(BULGE_URDF, rasterizer=oracle_rasterizer)
    # no stored pack and no URDF root: the error says what to pass
    with pytest.raises(FileNotFoundError, match='urdf_root'):
        PartPack.for_part(2, urdf_root=str(tmp_path))


def test_silhouette_march_rejects_bad_arguments():
    """Argument checks of `paintrl_silhouette_march` come before any CUDA call: testable without a GPU (-1 = PAINTRL_E_INVALID)."""
    import ctypes
    from paintrl_b200 import _capi
    lib = _capi.lib()
    n = np.array([[1.0, 0.0, 0.0]])
    off = np.array([1.0])
    pts = np.zeros((1, 3))
    mins = np.zeros(1, dtype=np.int8)
    out_b, out_f = np.zeros(1), np.zeros(1, dtype=np.int8)
    args = [n.ctypes.data, off.ctypes.data, 1, pts.ctypes.data, mins.ctypes.data, 1, 1, 0, 10, 0, out_b.ctypes.data, out_f.ctypes.data]
    bad_axes = list(args)
    bad_axes[6], bad_axes[7] = 2, 2                       # proof axis == non-principal axis
    assert lib.paintrl_silhouette_march(*bad_axes) == -1
    null_out = list(args)
    null_out[10] = None
    assert lib.paintrl_silhouette_march(*null_out) == -1
    no_planes = list(args)
    no_planes[2] = 0
    assert lib.paintrl_silhouette_march(*no_planes) == -1
    assert b'plane' in lib.paintrl_last_error() or b'null' in lib.paintrl_last_error()
