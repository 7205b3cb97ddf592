"""The scene description both the product and the oracle consume, checked against sources neither of them shares:
  * the compiled robot models (assets/*.agmodel.json, written by tools/compile_assets.py) against the reference's URDF files read
    with a separate, minimal XML walk (tests/golden/make_golden_reference_assets.py; its output is tests/golden/reference_assets.json);
  * masses, joint frames, axes and limits of the finalized scene arrays against the same XML;
  * inertia-from-shape of single primitives against the closed forms (sphere 2/5 m r^2; anything else: the box of the shape's
    bounding box, which is what Bullet's compound / createMultiBody path uses -- recalled, DESIGN.md section 5)."""
import json
import os

import numpy as np
import pytest

from assistive_gym_b200.scene import SceneBuilder

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROBOTS = ('jaco', 'pr2', 'sawyer')


def _stored_urdf_walk(name):
    """child link name -> (joint name, type, parent link, xyz, rpy, axis, lower, upper), link name -> (mass, com xyz, has <inertial>)"""
    u = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'reference_assets.json')))['urdf'][name]
    return u['joints'], u['links']


@pytest.mark.parametrize('name', ROBOTS)
def test_compiled_model_matches_the_urdf(name):
    joints, links = _stored_urdf_walk(name)
    m = json.load(open(os.path.join(ROOT, 'assistive_gym_b200', 'assets', name + '.agmodel.json')))
    assert len(m['links']) == len(links)
    seen = set()
    for k, lk in enumerate(m['links']):
        seen.add(lk['name'])
        mass, com, _ = links[lk['name']]
        assert abs(lk['inertial']['mass'] - mass) < 1e-12 and np.allclose(lk['inertial']['com_xyz'], com, atol=1e-12), lk['name']
        if lk['name'] not in joints:                      # the root link
            assert lk['parent'] < 0
            continue
        jn, jt, parent, xyz, rpy, axis, lo, hi = joints[lk['name']]
        j = lk['joint']
        assert j['name'] == jn and j['type'] == jt and m['links'][lk['parent']]['name'] == parent and lk['parent'] < k      # parents come first
        assert np.allclose(j['origin_xyz'], xyz, atol=1e-12) and np.allclose(j['origin_rpy'], rpy, atol=1e-12)
        if jt in ('revolute', 'continuous', 'prismatic'):
            assert np.allclose(j['axis'], axis, atol=1e-12)
        if jt in ('revolute', 'prismatic'):
            assert abs(j['lower'] - lo) < 1e-12 and abs(j['upper'] - hi) < 1e-12
    assert seen == set(links)


def test_scene_arrays_of_the_jaco_match_the_urdf():
    joints, links = _stored_urdf_walk('jaco')
    b = SceneBuilder()
    body = b.load_urdf('jaco', base_pos=[0.3, -0.1, 0.7], fixed_base=True)
    names = [lk.name for lk in b.links if lk.body == body]
    sc = b.finalize()
    l0 = int(sc['body_link0'][body])
    assert int(sc['body_nlinks'][body]) == len(links) == len(names)
    for i, nm in enumerate(names):
        k = l0 + i
        mass, com, has_inertial = links[nm]
        # a link without <inertial> gets Bullet's default mass 1 (its URDF importer's fallback); the base is held by `fixed_base`, whatever its mass
        assert abs(float(sc['link_mass'][k]) - (mass if has_inertial else 1.0)) < 1e-9, nm
        if nm not in joints:
            continue
        jn, jt, parent, xyz, rpy, axis, lo, hi = joints[nm]
        assert names[int(sc['link_parent'][k]) - l0] == parent
        assert np.allclose(sc['link_jpos'][k], xyz, atol=1e-9) and np.allclose(sc['link_com'][k], com, atol=1e-9)
        cr, sr, cp, sp_, cy, sy = np.cos(rpy[0]), np.sin(rpy[0]), np.cos(rpy[1]), np.sin(rpy[1]), np.cos(rpy[2]), np.sin(rpy[2])
        R = np.array([[cy * cp, cy * sp_ * sr - sy * cr, cy * sp_ * cr + sy * sr], [sy * cp, sy * sp_ * sr + cy * cr, sy * sp_ * cr - cy * sr], [-sp_, cp * sr, cp * cr]])
        x, y, z, w = sc['link_jquat'][k]
        Rq = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                       [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
        assert np.allclose(R, Rq, atol=1e-9)                                                 # URDF rpy = fixed-axis roll, pitch, yaw
        if jt in ('revolute', 'continuous'):
            assert np.allclose(sc['link_axis'][k], np.array(axis) / np.linalg.norm(axis), atol=1e-9)
        if jt == 'revolute':
            assert abs(float(sc['link_lower'][k]) - lo) < 1e-6 and abs(float(sc['link_upper'][k]) - hi) < 1e-6


@pytest.mark.parametrize('kind,kw,box', [
    ('sphere', dict(radius=0.07), None),
    ('box', dict(half_extents=[0.05, 0.12, 0.2]), [0.1, 0.24, 0.4]),
    ('capsule', dict(radius=0.04, height=0.3), [0.08, 0.08, 0.38]),          # along z, caps included
    ('cylinder', dict(radius=0.05, height=0.2), [0.1, 0.1, 0.2]),
])
def test_inertia_from_shape_closed_forms(kind, kw, box):
    mass = 1.7
    b = SceneBuilder()
    sh = b.create_collision_shape(kind, **kw)
    body = b.create_multibody(base_mass=mass, base_shape=sh, base_pos=[0, 0, 1])
    sc = b.finalize()
    k = int(sc['body_link0'][body])
    if box is None:
        want = np.full(3, 0.4 * mass * kw['radius'] ** 2)
    else:
        l = np.array(box)
        want = mass / 12.0 * np.array([l[1] ** 2 + l[2] ** 2, l[0] ** 2 + l[2] ** 2, l[0] ** 2 + l[1] ** 2])
    if kind == 'cylinder':                                    # a polygonal hull with a 1 mm rounding margin: its bounding box is 2 mm wider
        l = np.array(box) + 0.002
        want = mass / 12.0 * np.array([l[1] ** 2 + l[2] ** 2, l[0] ** 2 + l[2] ** 2, l[0] ** 2 + l[1] ** 2])
        assert np.allclose(sc['link_inertia'][k], want, rtol=2e-3)
        return
    assert np.allclose(sc['link_inertia'][k], want, rtol=1e-9, atol=1e-12)
