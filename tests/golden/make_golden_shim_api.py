"""Record how the UNMODIFIED reference SOT tracker (external/lib/test/tracker/unicorn_sot.py) uses the `unicorn` package, from the
imports to the point where it needs the GPU, as shim_sot_api.json: the names it imports from `unicorn`, the config file it asks
get_exp for, the Exp attributes it reads, the checkpoint key, and the model calls of its __init__ in order with their keyword
arguments.  tests/test_shim.py replays the record against unicorn_b200/shim.  Run where the reference checkout exists
(oracle/ref_import.REF_ROOT); the file is only parsed, not imported."""
import ast
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_import  # noqa: E402

SRC = "external/lib/test/tracker/unicorn_sot.py"
tree = ast.parse(open(os.path.join(ref_import.REF_ROOT, SRC)).read())
cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "UnicornSOTTrack")
init = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "__init__")


def is_self_model(node):
    return isinstance(node, ast.Attribute) and node.attr == "model" and isinstance(node.value, ast.Name) and node.value.id == "self"


def kwargs(call):
    return {k.arg: ast.literal_eval(k.value) for k in call.keywords if isinstance(k.value, ast.Constant)}


imports = sorted([n.module, a.name] for n in ast.walk(tree)
                 if isinstance(n, ast.ImportFrom) and n.module and n.module.split(".")[0] == "unicorn" for a in n.names)
exp_file = next(n.left.value for n in ast.walk(init)
                if isinstance(n, ast.BinOp) and isinstance(n.op, ast.Mod) and isinstance(n.left, ast.Constant) and "exps/" in n.left.value)
exp_attrs = sorted({n.attr for n in ast.walk(init) if isinstance(n, ast.Attribute) and isinstance(n.value, ast.Name) and n.value.id == "exp"})
get_model = next(n for n in ast.walk(init) if isinstance(n, ast.Call) and isinstance(n.func, ast.Attribute) and n.func.attr == "get_model")
ckpt_key = next(n.slice.value for n in ast.walk(init)
                if isinstance(n, ast.Subscript) and isinstance(n.value, ast.Call) and isinstance(n.value.func, ast.Attribute)
                and n.value.func.attr == "load" and isinstance(n.slice, ast.Constant))
model_calls = [[n.func.attr, kwargs(n)] for n in sorted((n for n in ast.walk(init) if isinstance(n, ast.Call)
                                                          and isinstance(n.func, ast.Attribute) and is_self_model(n.func.value)),
                                                         key=lambda n: (n.lineno, n.col_offset))]
model_attrs = sorted({n.attr for n in ast.walk(tree) if isinstance(n, ast.Attribute) and is_self_model(n.value)})

out = {"source": SRC, "imports": imports, "get_exp_file": exp_file, "exp_attributes": exp_attrs,
       "get_model_kwargs": kwargs(get_model), "checkpoint_key": ckpt_key, "init_model_calls": model_calls,
       "model_attributes": model_attrs}
with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "shim_sot_api.json"), "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out))
