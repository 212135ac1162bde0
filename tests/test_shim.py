"""The `unicorn`-importable shim (unicorn_b200/shim): API surface on CPU, and the UNMODIFIED reference tracker file
external/lib/test/tracker/unicorn_sot.py bound to the shim through its recorded use of the package (tests/golden/shim_sot_api.json,
written by tests/golden/make_golden_shim_api.py): its imports must resolve, its own __init__ sequence (get_exp -> get_model ->
torch.load -> load_state_dict) must run and stop exactly where the GPU is needed (`.cuda()`), with this package's loud
no-fallback error."""
import os
import subprocess
import sys
import textwrap

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
API = os.path.join(ROOT, "tests", "golden", "shim_sot_api.json")


def test_shim_surface():
    code = textwrap.dedent(f"""
        import sys
        sys.path.insert(0, {ROOT!r})
        import unicorn_b200.shim as shim
        shim.install()
        import torch
        from unicorn.exp import get_exp, ExpTrack
        from unicorn.utils import postprocess, fuse_model
        from unicorn.utils.boxes import postprocess_inst
        from unicorn.tracker.byte_tracker import BYTETracker, STrack
        from unicorn.tracker.quasi_dense_embed_tracker import QuasiDenseEmbedTracker
        from unicorn.models import Unicorn
        from unicorn_b200.weights import make_state_dict
        from unicorn_b200._lib import UnicornB200Error
        exp = get_exp("exps/default/unicorn_track_tiny_mask.py", None)
        assert exp.test_size == (800, 1280) and exp.normalize is False and exp.d_rate == 2 and exp.use_raft and exp.num_classes == 8
        exp.merge(["test_conf", "0.01"]); assert exp.test_conf == 0.01
        model = exp.get_model(load_pretrain=False)
        assert isinstance(model, Unicorn) and model.head.mask_head is not None and model.head.decode_in_inference
        sd = make_state_dict("unicorn_track_tiny_mask", 0)
        sd["head.mask_head._iter"] = torch.zeros(1)          # a buffer of the reference's DynamicMaskHead: tolerated
        r = model.load_state_dict(sd, strict=True)
        assert not r.missing_keys
        bad = dict(sd); bad.pop("head.stems.0.conv.weight")
        for strict in (True, False):
            try:
                model.load_state_dict(bad, strict=strict); raise SystemExit("missing key accepted")
            except RuntimeError:
                pass
        assert model.eval() is model and model.half() is model
        try:
            model(imgs=torch.zeros(1, 3, 32, 32), mode="backbone"); raise SystemExit("ran without a GPU engine")
        except RuntimeError:
            pass
        if not torch.cuda.is_available():
            try:
                model.cuda(); raise SystemExit("built an engine without a GPU")
            except UnicornB200Error:
                pass
        try:
            get_exp("exps/default/yolox_s.py", None); raise SystemExit("unknown config accepted")
        except KeyError:
            pass
        print("shim surface ok")
    """)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "shim surface ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.skipif(torch.cuda.is_available(), reason="on a GPU box the same flow runs to completion in tests/test_shim_gpu.py")
def test_unmodified_reference_sot_tracker_binds_to_shim(tmp_path):
    code = textwrap.dedent(f"""
        import importlib, json, sys
        sys.path.insert(0, {ROOT!r})
        import unicorn_b200.shim as shim
        shim.install()                                   # `unicorn` -> unicorn_b200/shim/unicorn
        import torch
        from unicorn_b200.weights import make_state_dict
        from unicorn_b200._lib import UnicornB200Error
        api = json.load(open({API!r}))
        names = {{}}
        for mod, name in api["imports"]:                 # the tracker file's `from unicorn... import ...` lines
            m = importlib.import_module(mod)
            assert m.__file__.startswith({os.path.join(ROOT, "unicorn_b200")!r}), (mod, m.__file__)
            names[name] = getattr(m, name)
        assert sys.modules["unicorn"].__unicorn_b200_shim__
        assert names["postprocess"].__module__ == "unicorn_b200.compat.model"
        ckpt = {str(tmp_path / 'c.pth')!r}
        torch.save({{api["checkpoint_key"]: make_state_dict("unicorn_track_tiny", 0)}}, ckpt)
        exp = names["get_exp"](api["get_exp_file"] % "unicorn_track_tiny", None)
        for a in api["exp_attributes"]:
            getattr(exp, a)
        model = exp.get_model(**api["get_model_kwargs"])
        missing = [a for a in api["model_attributes"] if not hasattr(model, a)]
        assert not missing, missing
        sd = torch.load(ckpt, map_location="cpu")[api["checkpoint_key"]]
        for meth, kw in api["init_model_calls"]:
            try:
                getattr(model, meth)(*((sd,) if meth == "load_state_dict" else ()), **kw)
            except UnicornB200Error as e:                # raised by self.model.cuda(): no CPU fallback
                assert meth == "cuda", meth
                print("stopped at .cuda():", str(e)[:80])
                break
        else:
            raise SystemExit("constructed without a GPU")
        print("reference tracker bound ok")
    """)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "reference tracker bound ok" in r.stdout, r.stdout + r.stderr
