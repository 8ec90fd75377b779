"""Do the reference's own scripts resolve against this repository?  (CPU; needs a checkout of the reference, named by
PAINTRL_REFERENCE: the scripts are not part of this repository.)

zigzag.py, spiral.py, paint_*.py and param_test_*.py import `PaintRLEnv.robot_gym_env.PaintGymEnv` /
`PaintRLEnv.param_test_env.ParamTestEnv` and drive them.  The scripts cannot be executed on the GPU box (the reference is
not there) nor here (no GPU), so this test reads them with `ast` and checks, name by name and call by call, that every
import from `PaintRLEnv.*`, every attribute used on the imported classes and on their instances, and every call's
argument list binds to what this repository exports under the same module path.  (The control loops themselves run on
the GPU in tests/test_gpu_gym_surface.py, re-typed from the scripts.)
"""
import ast
import importlib
import inspect
import os
import textwrap

import pytest

REF = os.environ.get('PAINTRL_REFERENCE', '')
SCRIPTS = ['zigzag.py', 'spiral.py', 'paint_ppo.py', 'param_test_ppo.py']
pytestmark = pytest.mark.skipif(not REF or not os.path.isfile(os.path.join(REF, 'zigzag.py')),
                                reason='PAINTRL_REFERENCE does not name a checkout of the reference')


def _calls_and_attributes(tree):
    """(imports {local name: (module, name)}, class-level attribute uses, instance attribute chains, calls)."""
    imports, class_attrs, inst_attrs, calls = {}, set(), set(), []
    for node in ast.walk(tree):
        if isinstance(node, ast.ImportFrom) and node.module and node.module.startswith('PaintRLEnv'):
            for a in node.names:
                imports[a.asname or a.name] = (node.module, a.name)
    instances = set()
    for node in ast.walk(tree):
        # `with Cls(...) as env:` / `env = Cls(...)`
        if isinstance(node, ast.With):
            for item in node.items:
                c = item.context_expr
                if isinstance(c, ast.Call) and isinstance(c.func, ast.Name) and c.func.id in imports and item.optional_vars is not None:
                    instances.add(item.optional_vars.id)
        if isinstance(node, ast.Assign) and isinstance(node.value, ast.Call) and isinstance(node.value.func, ast.Name) \
                and node.value.func.id in imports:
            for t in node.targets:
                if isinstance(t, ast.Name):
                    instances.add(t.id)

    def chain(n):
        parts = []
        while isinstance(n, ast.Attribute):
            parts.append(n.attr)
            n = n.value
        return (n.id, tuple(reversed(parts))) if isinstance(n, ast.Name) else (None, ())

    for node in ast.walk(tree):
        if isinstance(node, ast.Attribute):
            root, parts = chain(node)
            if root in imports:
                class_attrs.add((root, parts))
            elif root in instances:
                inst_attrs.add(parts)
        if isinstance(node, ast.Call):
            f = node.func
            root, parts = chain(f) if isinstance(f, ast.Attribute) else (f.id if isinstance(f, ast.Name) else None, ())
            if root in imports or root in instances:
                calls.append((root in imports, root, parts, len(node.args), [k.arg for k in node.keywords if k.arg],
                              any(k.arg is None for k in node.keywords)))
    return imports, class_attrs, inst_attrs, calls


def _instance_attributes(cls):
    """Names assigned on `self` anywhere in the class (and its bases in this repository) + class attributes."""
    names = set(dir(cls))
    for klass in cls.__mro__:
        try:
            src = inspect.getsource(klass)
        except (OSError, TypeError):
            continue
        for node in ast.walk(ast.parse(textwrap.dedent(src))):
            if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id == 'self' \
                    and isinstance(node.ctx, ast.Store):
                names.add(node.attr)
    return names


@pytest.mark.parametrize('script', SCRIPTS)
def test_script_resolves_against_this_repository(script):
    with open(os.path.join(REF, script)) as f:
        tree = ast.parse(f.read())
    imports, class_attrs, inst_attrs, calls = _calls_and_attributes(tree)
    assert imports, 'the script imports nothing from PaintRLEnv'
    resolved = {}
    for local, (module, name) in imports.items():
        mod = importlib.import_module(module)              # this repository's PaintRLEnv package
        assert os.path.realpath(mod.__file__).startswith(os.path.realpath(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))), mod.__file__
        assert hasattr(mod, name), '%s.%s' % (module, name)
        resolved[local] = getattr(mod, name)
    for root, parts in class_attrs:
        obj = resolved[root]
        for p in parts:
            assert hasattr(obj, p), '%s.%s (used by %s)' % (root, '.'.join(parts), script)
            obj = getattr(obj, p)
    for cls in resolved.values():
        have = _instance_attributes(cls)
        for parts in inst_attrs:
            assert parts[0] in have, 'instance attribute %s (used by %s)' % ('.'.join(parts), script)
    # `env.robot.reset(...)`: spiral.py:28-38 repositions the tool through the robot view
    if any(parts[:2] == ('robot', 'reset') for parts in inst_attrs):
        from paintrl_b200 import gym_env
        assert hasattr(gym_env._RobotView, 'reset')
    # every call binds: constructor, classmethods, step / reset
    for is_class, root, parts, n_pos, kw, star in calls:
        if is_class:
            target = resolved[root]
            for p in parts:
                target = getattr(target, p)
            sig = inspect.signature(target)
            if star:
                # `Cls(**env_config)` (paint_ppo.py:136, param_test_ppo.py:15): the dict literal that feeds it is the one
                # holding the constructor's first parameter; all of its keys must be constructor parameters
                first = next(iter(sig.parameters))
                dicts = [d for d in ast.walk(tree) if isinstance(d, ast.Dict) and any(
                    isinstance(k, ast.Constant) and k.value == first for k in d.keys)]
                assert dicts, (script, 'no env_config literal with %r' % first)
                for d in dicts:
                    keys = [k.value for k in d.keys if isinstance(k, ast.Constant)]
                    sig.bind(**{k: None for k in keys})
            else:
                sig.bind(*[None] * n_pos, **{k: None for k in kw})
        elif parts and parts[0] in ('step', 'reset'):
            for cls in resolved.values():
                sig = inspect.signature(getattr(cls, parts[0]))
                sig.bind(None, *[None] * n_pos, **{k: None for k in kw})


def test_wrapper_scripts_only_reexport():
    """paint_a3c.py ... param_test_impala.py are one-liners around paint_ppo.main / param_test_ppo.main."""
    for name in sorted(os.listdir(REF)):
        if name.endswith('.py') and name not in SCRIPTS:
            with open(os.path.join(REF, name)) as f:
                tree = ast.parse(f.read())
            mods = {n.module for n in ast.walk(tree) if isinstance(n, ast.ImportFrom)}
            assert mods <= {'paint_ppo', 'param_test_ppo'}, (name, mods)


def test_constructor_signature_matches_the_reference():
    """PaintGymEnv.__init__ / ParamTestEnv.__init__: same parameter names, order and defaults as the reference's source."""
    for module, cls_name in (('robot_gym_env', 'PaintGymEnv'), ('param_test_env', 'ParamTestEnv')):
        with open(os.path.join(REF, 'PaintRLEnv', module + '.py')) as f:
            tree = ast.parse(f.read())
        cls = next(n for n in ast.walk(tree) if isinstance(n, ast.ClassDef) and n.name == cls_name)
        init = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == '__init__')
        ref_names = [a.arg for a in init.args.args]
        ref_defaults = [ast.literal_eval(d) for d in init.args.defaults]
        ours = inspect.signature(getattr(importlib.import_module('PaintRLEnv.' + module), cls_name).__init__)
        our_params = list(ours.parameters.values())
        assert [p.name for p in our_params][:len(ref_names)] == ref_names, (cls_name, [p.name for p in our_params], ref_names)
        with_default = [p.default for p in our_params[:len(ref_names)] if p.default is not inspect.Parameter.empty]
        assert with_default == ref_defaults, (cls_name, with_default, ref_defaults)
