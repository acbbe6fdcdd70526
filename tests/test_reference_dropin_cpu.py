"""Drop-in check of the registry boundary: `register_into_reference()` must make the reference's OWN registries build the
esb200 classes from the reference's UNMODIFIED config files. tests/golden/dropin.json (make_golden.py dropin) holds the
`model` dicts of those config files and the names the reference's registries hold once its models are imported; the
registries are rebuilt here as `embodiedscan/registry.py` defines them, every one of those names already taken, so the
test needs neither the reference tree nor its third-party stack."""
import ast
import json
import os
import sys
import types

import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
with open(os.path.join(GOLD, 'dropin.json')) as _f:
    DROPIN = json.load(_f)


def reference_registry_module(monkeypatch):
    """`embodiedscan.registry`: MODELS and TASK_UTILS as children of mmengine's roots (the mmengine stand-in of
    refstubs.py), each holding a class of the reference under every name the reference registers."""
    if GOLD not in sys.path:
        sys.path.insert(0, GOLD)
    from refstubs import Registry
    mod = types.ModuleType('embodiedscan.registry')
    for attr, key in (('MODELS', 'models'), ('TASK_UTILS', 'task_utils')):
        reg = Registry(attr.lower(), parent=Registry(attr.lower()))
        for name in DROPIN[key]:
            reg.register_module(module=type(name, (), {'__module__': 'embodiedscan.models'}))
        setattr(mod, attr, reg)
    pkg = types.ModuleType('embodiedscan')
    pkg.__path__, pkg.registry = [], mod
    monkeypatch.setitem(sys.modules, 'embodiedscan', pkg)
    monkeypatch.setitem(sys.modules, 'embodiedscan.registry', mod)
    return mod


@pytest.mark.parametrize('cfg_file,cls_name', [
    ('configs/detection/mv-det3d_8xb4_embodiedscan-3d-284class-9dof.py', 'SparseFeatureFusionSingleStage3DDetector'),
    ('configs/detection/cont-det3d_8xb1_embodiedscan-3d-284class-9dof.py', 'Embodied3DDetector'),
    ('configs/occupancy/mv-occ_8xb1_embodiedscan-occ-80class.py', 'DenseFusionOccPredictor'),
    ('configs/occupancy/cont-occ_8xb1_embodiedscan-occ-80class.py', 'EmbodiedOccPredictor'),
    ('configs/grounding/mv-grounding_8xb12_embodiedscan-vg-9dof.py', 'SparseFeatureFusion3DGrounder'),
    ('configs/grounding/mv-grounding_8xb12_embodiedscan-vg-9dof_fcaf-coder.py', 'SparseFeatureFusion3DGrounder'),
])
def test_reference_registry_builds_esb200_from_unmodified_configs(cfg_file, cls_name, monkeypatch):
    ref = reference_registry_module(monkeypatch)
    assert cls_name in DROPIN['models']                   # the reference's own class holds the name until the override

    import embodiedscan_b200
    from embodiedscan_b200.registry import register_into_reference
    register_into_reference()
    model_cfg = ast.literal_eval(DROPIN['configs'][cfg_file])
    assert model_cfg['type'] == cls_name
    for sub in ('backbone', 'neck'):                      # pretrained-checkpoint URLs need a network
        if isinstance(model_cfg.get(sub), dict):
            model_cfg[sub].pop('init_cfg', None)
    model = ref.MODELS.build(model_cfg)
    assert type(model).__module__.startswith('embodiedscan_b200'), type(model)
    assert type(model) is getattr(embodiedscan_b200, cls_name, None) or type(model).__name__ == cls_name
    names = dict(model.named_parameters())
    assert any(k.endswith('.kernel') for k in names) and 'backbone_3d.conv1.kernel' in names
