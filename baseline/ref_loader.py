"""Import the UNMODIFIED reference from oracle/_ref (installed by oracle/install_reference.py).  Test / bench
infrastructure only - nothing under must3r_b200/ imports this.

    ref = load_reference(curope_shim=False)     # -> namespace with .model, .engine, .Dust3rEncoder, .MUSt3R
    ref = load_reference(curope_shim=True)      # reference RoPE served by must3r_b200.compat.curope (CUDA only)

The RoPE implementation is chosen by the reference at import time (pos_embed.py:104-110), so the choice is per process:
a second call with a different `curope_shim` raises.
"""
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(os.path.dirname(HERE), "oracle", "_ref")
_loaded = {}


def available():
    return os.path.isdir(os.path.join(REF, "must3r")) and os.path.isdir(os.path.join(REF, "dust3r", "dust3r"))


def load_reference(curope_shim=False, quiet=True):
    if "ns" in _loaded:
        if _loaded["shim"] != curope_shim:
            raise RuntimeError("the reference was already imported with curope_shim=%s in this process" % _loaded["shim"])
        return _loaded["ns"]
    if not available():
        raise ImportError("oracle/_ref is missing: run oracle/install_reference.py <checkout of the reference>")
    if REF not in sys.path:
        sys.path.insert(0, REF)
    stubs = os.path.join(HERE, "stubs")
    if stubs not in sys.path:
        sys.path.append(stubs)                     # `roma` placeholder, found only if the real one is absent
    if curope_shim:
        root = os.path.dirname(HERE)
        if root not in sys.path:
            sys.path.insert(0, root)
        import must3r_b200.compat.curope as shim
        sys.modules["curope"] = shim
    else:
        assert "curope" not in sys.modules, "a curope module is already imported: the reference would silently pick it"
    import contextlib
    import io
    with (contextlib.redirect_stdout(io.StringIO()) if quiet else contextlib.nullcontext()):
        import must3r.model as model
        import must3r.engine.inference as engine
        from must3r.model.blocks import attention as attn_mod
        import models.pos_embed as pe                # croco's module, aliased by path_to_croco
    ns = types.SimpleNamespace(model=model, engine=engine, attention=attn_mod, Dust3rEncoder=model.Dust3rEncoder,
                               MUSt3R=model.MUSt3R, rope_class=pe.RoPE2D.__name__, pos_embed=pe)
    if curope_shim:
        assert pe.RoPE2D.__name__ == "cuRoPE2D", "the reference did not pick up the curope shim"
    else:
        assert pe.RoPE2D.__name__ == "RoPE2D", "the reference picked a native curope although none was requested"
    _loaded.update(ns=ns, shim=curope_shim)
    return ns
