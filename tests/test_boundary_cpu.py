"""Drop-in boundary, host side (SURVEY.md section 8b): every name the reference's eval scripts import from the `groma` package
exists in this repo's `groma` package, the scripts' module bodies execute on top of it, `model.generation_config` carries the
checkpoint's EOS / pad ids, and `AutoModel.from_pretrained` resolves to GromaModel.  No GPU needed.

What the scripts' module bodies execute -- their import statements and the base classes of the classes they define -- is
stored in tests/golden/eval_script_imports.json (tests/golden/make_eval_imports_golden.py)."""
import ast
import importlib
import json
import os
import sys
import types

import pytest
import torch

SCRIPTS = ["run_groma.py", "run_ddetr.py", "eval_rec.py", "eval_lvis.py", "model_vg.py", "model_refcocog.py", "model_vqa.py"]
# modules of the reference's `groma` package that are on the path and therefore provided by this repo
PROVIDED = {"groma.utils", "groma.constants", "groma.model.groma", "groma.model.ddetr", "groma.data.conversation"}
with open(os.path.join(os.path.dirname(__file__), "golden", "eval_script_imports.json")) as _f:
    EVAL_SCRIPTS = json.load(_f)


def _groma_imports(script):
    for st in EVAL_SCRIPTS[script]["imports"]:
        if st.get("from") and st["from"].startswith("groma"):
            yield st["from"], [n for n, _ in st["names"]]


def _import_node(st):
    if "import" in st:
        return ast.Import(names=[ast.alias(name=n, asname=a) for n, a in st["import"]])
    return ast.ImportFrom(module=st["from"], names=[ast.alias(name=n, asname=a) for n, a in st["names"]], level=st["level"])


@pytest.mark.parametrize("script", SCRIPTS)
def test_names_the_eval_scripts_import_exist(script):
    for mod, names in _groma_imports(script):
        if mod not in PROVIDED:
            assert mod.startswith("groma.data.datasets"), f"{script} imports {mod}, which is neither provided nor a dataset module"
            continue
        m = importlib.import_module(mod)
        for n in names:
            assert hasattr(m, n), f"{script}: `from {mod} import {n}` would fail"


class _Anything(types.ModuleType):
    """Stand-in for a third-party / dataset module that is absent in this image: CamelCase attributes are empty base
    classes (the scripts subclass dataset classes), everything else a dummy callable."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        if name[0].isupper() and not name.isupper():
            return type(name, (), {})
        return lambda *a, **k: None


@pytest.mark.parametrize("script", SCRIPTS)
def test_eval_script_module_bodies_execute_on_this_package(script, monkeypatch):
    """Execute what the reference script's module body executes (its imports, and the base classes of the classes it defines;
    its functions take no defaults or decorators, and `__main__` does not run) with `groma.*` resolving to THIS repo; only
    packages missing from the image (mmcv, mmdet, pycocotools, lvis) and the dataset modules are stood in for."""
    body = EVAL_SCRIPTS[script]
    absent_roots = {"mmcv", "mmdet", "pycocotools", "lvis"}
    for st in body["imports"]:
        mods = [n for n, _ in st["import"]] if "import" in st else [st["from"]] if st["from"] else []
        for mod in mods:
            if mod.split(".")[0] in absent_roots or mod.startswith("groma.data.datasets"):
                parts = mod.split(".")
                for i in range(1, len(parts) + 1):
                    name = ".".join(parts[:i])
                    if name not in sys.modules and not name == "groma" and not name == "groma.data":
                        monkeypatch.setitem(sys.modules, name, _Anything(name))
    ns = {"__name__": "ref_eval_" + script[:-3]}
    module = ast.fix_missing_locations(ast.Module(body=[_import_node(st) for st in body["imports"]], type_ignores=[]))
    exec(compile(module, script, "exec"), ns)
    for base in body["class_bases"]:
        assert isinstance(eval(base, ns), type), f"{script}: base class {base} does not resolve"
    import groma.model.groma as ours
    if "GromaModel" in ns:
        assert ns["GromaModel"] is ours.GromaModel
    if "init_distributed_mode" in ns:
        import groma.utils
        assert ns["init_distributed_mode"] is groma.utils.init_distributed_mode


def test_init_distributed_mode_without_launcher_env(monkeypatch):
    from groma.utils import init_distributed_mode
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "SLURM_PROCID"):
        monkeypatch.delenv(k, raising=False)
    args = types.SimpleNamespace()
    init_distributed_mode(args)
    assert args.distributed is False


def test_generation_config_from_checkpoint_dir(tmp_path):
    """train.py:108-112 writes eos / pad / bos into generation_config.json; run_groma.py:92 passes it back to generate()."""
    from groma.model.groma import GromaConfig, _eos_list, _load_generation_config
    from groma_b200.config import tiny_config
    cfg = GromaConfig.from_path_config(tiny_config())
    gc = _load_generation_config(None, cfg)                      # no file: ids from llm_cfg (LlamaConfig defaults 2 / 1)
    assert gc.eos_token_id == cfg.llm_cfg.eos_token_id and gc.bos_token_id == cfg.llm_cfg.bos_token_id
    (tmp_path / "generation_config.json").write_text(json.dumps({"eos_token_id": [2, 7], "pad_token_id": 1000, "bos_token_id": 1,
                                                                 "do_sample": True, "max_new_tokens": 33}))
    gc = _load_generation_config(str(tmp_path), cfg)
    assert _eos_list(gc.eos_token_id) == [2, 7] and gc.pad_token_id == 1000 and gc.max_new_tokens == 33
    assert _eos_list(None) == [] and _eos_list(5) == [5] and _eos_list(torch.tensor([3, 4])) == [3, 4]


def test_automodel_resolves_groma_model(tmp_path):
    """AutoConfig / AutoModel registration (reference groma.py:430-431): AutoModel.from_pretrained(dir) must land in
    GromaModel.from_pretrained with the parsed GromaConfig -- observed here through the loader's own error for a weightless dir."""
    from transformers import AutoConfig, AutoModel
    import groma.model.groma as gm
    from groma_b200.config import tiny_config
    gm.GromaConfig.from_path_config(tiny_config()).save_pretrained(str(tmp_path))
    assert isinstance(AutoConfig.from_pretrained(str(tmp_path)), gm.GromaConfig)
    with pytest.raises(FileNotFoundError, match="safetensors"):
        AutoModel.from_pretrained(str(tmp_path))
