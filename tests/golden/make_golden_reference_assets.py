"""What the asset tests need from the reference's own asset files, so that they run without the reference checkout:
  * the three robot URDFs read with a minimal XML walk of their own (not tools/compile_assets.py): per joint (name, type,
    parent link, origin xyz / rpy, axis, limits), per link (mass, com, whether it has an <inertial>)
    -> reference_assets.json['urdf'] (tests/test_scene_description.py);
  * clothing/hospitalgown_reduced.obj: the number of its `v` lines and, in `v`-line order, the vertices at the node indices of the
    two sleeve triangles (dressing.py:149-150) -> reference_assets.json['gown_obj'] (tests/test_cloth_model.py);
  * realistic_arm_limits_model.h5, copied unchanged: the input of the HDF5 reader in tools/compile_assets.py
    (tests/test_env_surface.py).

usage: python tests/golden/make_golden_reference_assets.py [/root/reference]"""
import json
import os
import shutil
import sys
import xml.etree.ElementTree as ET

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from assistive_gym_b200.dressing_batch import TRIANGLE1, TRIANGLE2  # noqa: E402

URDFS = {'jaco': 'jaco/j2s7s300_gym.urdf', 'sawyer': 'sawyer/sawyer.urdf', 'pr2': 'PR2/pr2_no_torso_lift_tall.urdf'}


def _floats(s, n, default=0.0):
    v = [float(x) for x in s.split()] if s else []
    return v + [default] * (n - len(v))


def walk_urdf(path):
    """child link name -> (joint name, type, parent link, xyz, rpy, axis, lower, upper), link name -> (mass, com xyz, has <inertial>)"""
    root = ET.parse(path).getroot()
    joints, links = {}, {}
    for j in root.findall('joint'):
        o, a, lim = j.find('origin'), j.find('axis'), j.find('limit')
        joints[j.find('child').get('link')] = (
            j.get('name'), j.get('type'), j.find('parent').get('link'),
            _floats(o.get('xyz') if o is not None else '', 3), _floats(o.get('rpy') if o is not None else '', 3),
            _floats(a.get('xyz'), 3) if a is not None else [1.0, 0.0, 0.0],
            float(lim.get('lower', 0.0)) if lim is not None else 0.0, float(lim.get('upper', 0.0)) if lim is not None else 0.0)
    for l in root.findall('link'):
        i = l.find('inertial')
        m, c = 0.0, [0.0, 0.0, 0.0]
        if i is not None:
            m = float(i.find('mass').get('value'))
            o = i.find('origin')
            c = _floats(o.get('xyz') if o is not None else '', 3)
        links[l.get('name')] = (m, c, i is not None)
    return joints, links


def main():
    ref = sys.argv[1] if len(sys.argv) > 1 else '/root/reference'
    assets = os.path.join(ref, 'assistive_gym', 'envs', 'assets')
    out = {'urdf': {}}
    for name, rel in sorted(URDFS.items()):
        joints, links = walk_urdf(os.path.join(assets, rel))
        out['urdf'][name] = {'joints': joints, 'links': links}
    v = [[float(t) for t in l.split()[1:4]] for l in open(os.path.join(assets, 'clothing', 'hospitalgown_reduced.obj')) if l.startswith('v ')]
    idx = TRIANGLE1 + TRIANGLE2
    out['gown_obj'] = {'n_vertices': len(v), 'indices': idx, 'vertices': [v[i] for i in idx]}
    with open(os.path.join(HERE, 'reference_assets.json'), 'w') as f:
        json.dump(out, f, sort_keys=True)
    shutil.copyfile(os.path.join(assets, 'realistic_arm_limits_model.h5'), os.path.join(HERE, 'realistic_arm_limits_model.h5'))
    print(' | '.join('%s: %d links %d joints' % (k, len(u['links']), len(u['joints'])) for k, u in out['urdf'].items()),
          '| gown obj: %d vertices' % len(v))


if __name__ == '__main__':
    main()
