"""Check of the drop-in surface (SURVEY 8b): every call the original project's orchestration (pipelines/pipeline.py)
makes on the hot-path objects, and every constructor parameter its shipped pipeline factories can pass, exists on the
engine's classes with a compatible signature.  The surface is stored in tests/golden/reference_surface.json.  Where
the original sources are available, the stored sets are also checked against them.  The calls themselves are
exercised on the GPU by tests/test_gpu_host_api.py::test_train_checkpoint_resume_through_the_reference_protocol.
"""
import ast
import inspect
import json
import os

import pytest

import ref_shims

COMPONENT_CLASSES = {
    "policy": ("GaussianActor_NeuralNetwork", "GaussianActorCritic_NeuralNetwork"),
    "algorithm": ("GRPO", "PPO"),
    "buffer": ("Rollout_Buffer",),
    "rollout_manager": ("RolloutManager",),
}
FACTORIES = ["cartpole_pipeline_grpo", "cartpole_pipeline_ppo", "quadpole2d_pipeline_ppo", "quadpole_pipeline_ppo"]


@pytest.fixture(scope="module")
def surface(golden_dir):
    with open(os.path.join(golden_dir, "reference_surface.json")) as f:
        return json.load(f)


def _calls_on_components(tree):
    """{component: {(method, n_args), ...}} for every `self.<component>.<method>(...)` in the reference Pipeline."""
    found = {}
    for node in ast.walk(tree):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute):
            inner = node.func.value
            if isinstance(inner, ast.Attribute) and isinstance(inner.value, ast.Name) and inner.value.id == "self":
                found.setdefault(inner.attr, set()).add((node.func.attr, len(node.args)))
    return found


def _factory_keywords(tree, names):
    """{class name: {keyword, ...}} of the constructor calls in a reference pipeline factory."""
    found = {}
    for node in ast.walk(tree):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Name) and node.func.id in names:
            found.setdefault(node.func.id, set()).update(kw.arg for kw in node.keywords)
    return found


def _init_params(cls):
    return list(inspect.signature(cls.__init__).parameters.values())[1:]


def test_reference_pipeline_calls_exist_on_engine_classes(surface):
    import trajopt_grpo_b200 as tg
    calls = {comp: {tuple(c) for c in cs} for comp, cs in surface["pipeline_calls"].items()}
    if ref_shims.available():
        with open(os.path.join(ref_shims.REFERENCE_ROOT, "pipelines", "pipeline.py")) as f:
            parsed = _calls_on_components(ast.parse(f.read()))
        for comp in COMPONENT_CLASSES:
            assert parsed.get(comp, set()) <= calls[comp], (comp, parsed.get(comp, set()) - calls[comp])
    assert {"policy", "algorithm", "buffer", "rollout_manager"} <= set(calls)
    for comp, classes in COMPONENT_CLASSES.items():
        for meth, nargs in calls[comp]:
            for cname in classes:
                cls = getattr(tg, cname)
                assert hasattr(cls, meth), f"reference Pipeline calls {comp}.{meth}() but {cname} has no such method"
                sig = inspect.signature(getattr(cls, meth))
                required = [p for p in list(sig.parameters.values())[1:] if p.default is p.empty
                            and p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]
                assert len(required) <= nargs <= len(sig.parameters) - 1, (cname, meth, nargs, str(sig))


@pytest.mark.parametrize("cname", ["GaussianActor_NeuralNetwork", "GaussianActorCritic_NeuralNetwork", "GRPO", "PPO",
                                   "RolloutManager", "Rollout_Buffer", "CartPole", "Pendulum", "QuadPole2D", "QuadPole"])
def test_reference_constructor_parameters_accepted_by_engine_classes(surface, cname):
    """Every keyword the shipped pipeline factories (pipelines/*_pipeline_*.py:54-80) can pass to this constructor is
    accepted by the engine's class; where the original signature is stored, positional arguments bind to the same
    parameters and the engine requires none that the original does not."""
    import trajopt_grpo_b200 as tg
    ref = surface["constructors"][cname]
    accepted = ref.get("positional", []) + ref.get("keywords", [])
    if ref_shims.available():
        for factory in FACTORIES:
            path = os.path.join(ref_shims.REFERENCE_ROOT, "pipelines", factory + ".py")
            if os.path.exists(path):
                with open(path) as f:
                    used = _factory_keywords(ast.parse(f.read()), {cname}).get(cname, set())
                assert used <= set(accepted), (factory, cname, used - set(accepted))
    params = _init_params(getattr(tg, cname))
    names = [p.name for p in params if p.kind in (p.POSITIONAL_OR_KEYWORD, p.KEYWORD_ONLY)]
    for kw in accepted:
        assert kw in names, f"{cname}({kw}=...) is not accepted by the engine's class"
    if "positional" in ref:
        pos = [p for p in params if p.kind == p.POSITIONAL_OR_KEYWORD]
        assert [p.name for p in pos[:len(ref["positional"])]] == ref["positional"], (cname, [p.name for p in pos])
        assert sum(p.default is p.empty for p in pos) <= ref["required"], cname
        assert all(p.default is not p.empty for p in params if p.kind == p.KEYWORD_ONLY), cname
