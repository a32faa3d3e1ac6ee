"""Drop-in boundary against the REAL caller (SURVEY.md 7 step 2c): the reference's own, unmodified `src/model.py` is
imported from the RWKV_LM_EXT checkout named by $RWKV_LM_EXT_SRC (skipped without one) -- with its working directory
pointing at shim/ (whose cuda/*_op.cpp replace the reference's), so that ITS `load(name="wkv6", sources=["cuda/wkv6_op.cpp",
"cuda/wkv6_cuda.cu"], ...)` call (src/model.py:188-189) builds and imports OUR module; then `rwkv_lm_ext_b200.install`
repoints the module-level operator every `RWKV_Tmix_x060` layer calls.  No GPU needed: nothing is launched."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("RWKV_LM_EXT_SRC", "")        # an unmodified checkout of yynil/RWKV_LM_EXT

_SCRIPT = textwrap.dedent(r"""
    import os, sys, types
    ROOT, REF = sys.argv[1], sys.argv[2]
    # the two stubs of SURVEY.md 8(c): Lightning and bitsandbytes are not installed here and not on the path under test
    pl = types.ModuleType("pytorch_lightning"); pl.__version__ = "2.0"
    import torch.nn as nn
    pl.LightningModule = type("LightningModule", (nn.Module,), {})
    pl.Callback = object
    ut = types.ModuleType("pytorch_lightning.utilities"); ut.rank_zero_info = print; ut.rank_zero_only = lambda f: f
    st = types.ModuleType("pytorch_lightning.strategies"); st.DeepSpeedStrategy = type("DeepSpeedStrategy", (), {})
    sys.modules.update({"pytorch_lightning": pl, "pytorch_lightning.utilities": ut, "pytorch_lightning.strategies": st,
                        "bitsandbytes": types.ModuleType("bitsandbytes")})
    os.environ.update(WKV="", RWKV_TRAIN_TYPE=os.environ.get("TT", ""), RWKV_MY_TESTING="x060", RWKV_JIT_ON="0", RWKV_HEAD_SIZE_A="64",
                      RWKV_CTXLEN="4096", RWKV_FLOAT_MODE="bf16", RWKV_T_MAX="4096", TORCH_CUDA_ARCH_LIST="10.0",
                      TORCH_EXTENSIONS_DIR=os.path.join(ROOT, "shim", "_build", "_jit"))
    sys.path.insert(0, REF)
    sys.path.insert(0, ROOT)
    os.chdir(os.path.join(ROOT, "shim"))          # src/model.py names its sources relative to the working directory
    import src.model as m                          # the reference, unmodified: runs its load() on shim/cuda/*
    import rwkv_lm_ext_b200 as wkv
    if os.environ.get("TT") == "infctx":
        mod = m.wkv6state_cuda
        assert "libwkv6_b200" in mod.forward.__doc__ and mod.__name__ == "wkv6infctx", mod
    else:
        mod = m.wkv6_cuda
        assert "libwkv6_b200" in mod.forward.__doc__ and "libwkv6_b200" in mod.backward.__doc__, mod.forward.__doc__
        assert m.WKV_6.forward.__globals__["wkv6_cuda"] is mod          # the reference's autograd Function calls our module
        ref_run = m.RUN_CUDA_RWKV6
        wkv.install(m)
        assert m.RUN_CUDA_RWKV6 is wkv.RUN_CUDA_RWKV6 and m.RUN_CUDA_RWKV6 is not ref_run
        # every time-mix layer resolves the operator through the module globals at call time
        fwd = m.RWKV_Tmix_x060.forward
        assert fwd.__globals__["RUN_CUDA_RWKV6"] is wkv.RUN_CUDA_RWKV6
        assert "RUN_CUDA_RWKV6" in fwd.__code__.co_names
    print("INTEGRATION_OK", mod.__file__)
""")


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "src")),
                    reason="needs an unmodified RWKV_LM_EXT checkout: set RWKV_LM_EXT_SRC to its directory")
@pytest.mark.parametrize("train_type", ["", "infctx"])
def test_unmodified_reference_model_loads_our_ops(tmp_path, train_type):
    script = tmp_path / "probe.py"
    script.write_text(_SCRIPT)
    env = dict(os.environ, TT=train_type)
    out = subprocess.run([sys.executable, str(script), ROOT, REF], capture_output=True, text=True, timeout=900, env=env)
    assert "INTEGRATION_OK" in out.stdout, out.stdout[-3000:] + "\n" + out.stderr[-3000:]


def test_shim_sources_cover_every_reference_module():
    """One *_op.cpp + the source file name the reference's load() lists next to it, per native module (SURVEY.md 8b)."""
    want = {"wkv6_op.cpp", "wkv6_cuda.cu", "wkv6state_op.cpp", "wkv6state_cuda.cu", "wkv6infctx_op.cpp", "wkv6infctx_cuda.cu",
            "wkv6_bi_op.cpp", "wkv6_bi_cuda.cu", "rwkv6_op.cpp", "rwkv6.cu"}
    have = set(os.listdir(os.path.join(ROOT, "shim", "cuda")))
    assert want <= have
    for f in want:
        if f.endswith("_op.cpp"):
            src = open(os.path.join(ROOT, "shim", "cuda", f)).read()
            assert "PYBIND11_MODULE" in src and "wkv6_b200_dl.h" in src
