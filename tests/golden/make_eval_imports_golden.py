"""Generate tests/golden/eval_script_imports.json: for each of the REFERENCE's eval scripts (groma/eval/*.py) the import
statements its module body executes and the base classes of the classes it defines, as data (module and name lists, no
source text).  tests/test_boundary_cpu.py replays them against this repo's `groma` package; the reference is not part of
this repository, hence the committed fixture.

    python -m tests.golden.make_eval_imports_golden <reference checkout>"""
import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SCRIPTS = ["run_groma.py", "run_ddetr.py", "eval_rec.py", "eval_lvis.py", "model_vg.py", "model_refcocog.py", "model_vqa.py"]


def describe(path):
    tree = ast.parse(open(path).read())
    imports, bases = [], []
    for n in tree.body:
        if isinstance(n, ast.Import):
            imports.append({"import": [[a.name, a.asname] for a in n.names]})
        elif isinstance(n, ast.ImportFrom):
            imports.append({"from": n.module, "level": n.level, "names": [[a.name, a.asname] for a in n.names]})
        elif isinstance(n, ast.ClassDef):
            bases += [ast.unparse(b) for b in n.bases]
        elif isinstance(n, ast.FunctionDef):
            assert not n.decorator_list and not n.args.defaults and not any(n.args.kw_defaults), f"{path}: {n.name}"
        elif not (isinstance(n, ast.If) and ast.unparse(n.test) == "__name__ == '__main__'"):
            raise ValueError(f"{path}: module-level {type(n).__name__} is not described by this fixture")
    nested = [n for n in ast.walk(tree) if isinstance(n, (ast.Import, ast.ImportFrom))]
    assert len(nested) == len(imports), f"{path}: imports outside the module body"
    return {"imports": imports, "class_bases": bases}


if __name__ == "__main__":
    eval_dir = os.path.join(sys.argv[1], "groma", "eval")
    out = {s: describe(os.path.join(eval_dir, s)) for s in SCRIPTS}
    blocks = []
    for s, d in out.items():        # one import statement per line
        imports = ",\n".join("   " + json.dumps(i) for i in d["imports"])
        blocks.append(f' {json.dumps(s)}: {{\n  "imports": [\n{imports}\n  ],\n  "class_bases": {json.dumps(d["class_bases"])}\n }}')
    with open(os.path.join(HERE, "eval_script_imports.json"), "w") as f:
        f.write("{\n" + ",\n".join(blocks) + "\n}\n")
    assert json.load(open(os.path.join(HERE, "eval_script_imports.json"))) == out
    print("wrote eval_script_imports.json")
