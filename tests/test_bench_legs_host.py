"""test_gpu_bench_legs.py replays bench.py's legs in process; this checks, from bench.py's source, that the replay drives the
plan as bench.py does: the PlanConfig keywords of make_plan, the push size rule, the seed of each IF's input and the plan
calls of a timed step and of an e2e step.  If bench.py changes how it drives the plan, the test names what changed."""
import ast
import os

import test_gpu_bench_legs as legs

BENCH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")


def _tree():
    with open(BENCH) as f:
        return ast.parse(f.read())


def _func(node, name):
    for n in ast.walk(node):
        if isinstance(n, ast.FunctionDef) and n.name == name:
            return n
    raise AssertionError(f"bench.py has no function {name}")


def _calls(node):
    out = [n for n in ast.walk(node) if isinstance(n, ast.Call)]
    return sorted(out, key=lambda c: (c.lineno, c.col_offset))


def _call_name(c):
    f = c.func
    return f.attr if isinstance(f, ast.Attribute) else f.id if isinstance(f, ast.Name) else None


def _make_plan_args(main):
    """third argument of every make_plan(...) call in main, by the name it is assigned to"""
    out = {}
    for n in ast.walk(main):
        if isinstance(n, ast.Assign) and isinstance(n.value, ast.Call) and _call_name(n.value) == "make_plan":
            out[n.targets[0].id] = ast.unparse(n.value.args[2])
    return out


def test_plan_keywords():
    make_plan = _func(_func(_tree(), "main"), "make_plan")
    cfg = [c for c in _calls(make_plan) if _call_name(c) == "PlanConfig"]
    assert len(cfg) == 1
    assert tuple(k.arg for k in cfg[0].keywords) == legs.PLAN_KEYWORDS


def test_chunk_unit_rule():
    tree = _tree()
    args = _make_plan_args(_func(tree, "main"))
    assert args["pl"] == legs.CHUNK_UNITS_RULE
    assert args["pls"] == legs.STRONG_CHUNK_UNITS_RULE
    default = [c for c in _calls(tree) if _call_name(c) == "add_argument" and ast.literal_eval(c.args[0]) == "--chunk-units"]
    assert len(default) == 1
    assert ast.literal_eval([k.value for k in default[0].keywords if k.arg == "default"][0]) == legs.BENCH_CHUNK_UNITS


def test_device_seed():
    main = _func(_tree(), "main")
    seeds = [ast.unparse(c.args[3]) for c in _calls(main) if _call_name(c) == "make_device_vdif"]
    assert seeds == [legs.SEED_RULE]


def _plan_calls(fn, plan_names):
    out = []
    for c in _calls(fn):
        f = c.func
        if isinstance(f, ast.Attribute) and isinstance(f.value, ast.Name) and f.value.id in plan_names:
            if f.attr == "push":
                kw = {k.arg: ast.literal_eval(k.value) for k in c.keywords if k.arg == "on_device"}
                out.append(f"push(on_device={kw.get('on_device')})")
            else:
                out.append(f.attr)
        elif _call_name(c) == "b2f_push":
            out.append(f"b2f_push(..., {ast.unparse(c.args[-1])})")
    return tuple(out)


def test_step_calls():
    main = _func(_tree(), "main")
    assert _plan_calls(_func(_func(main, "make_step"), "step"), {"plan"}) == legs.DEVICE_STEP_CALLS
    assert _plan_calls(_func(main, "step_host"), {"pl"}) == legs.HOST_STEP_CALLS
