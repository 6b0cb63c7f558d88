"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every
symbol include/l2s_vocoder.h declares, validates configs without touching CUDA,
and the host classes keep the reference's surface.  No compute call is made."""
import ctypes as C
import os
import re

import pytest
import torch
import torch.multiprocessing as mp

from oracle import vocoder_oracle as vo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(pkg):
    lib = pkg._cabi.load()
    text = ""
    for name in ("l2s_vocoder.h", "l2s_debug.h", "l2s_hand_off.h"):       # the drop-in boundary, the test hooks, the hand-off file I/O
        with open(os.path.join(ROOT, "include", name)) as f:
            text += f.read()
    declared = set(re.findall(r"\b(l2s_[a-z0-9_]+)\s*\(", text))
    assert declared, "no prototypes found in the header"
    assert declared == set(pkg._cabi.EXPORTS)
    for sym in declared:
        assert getattr(lib, sym) is not None
    assert b"sm_100a" in lib.l2s_version()


def _cfg(pkg, **over):
    h = pkg.AttrDict(vo.shipped_config(**over))
    g = pkg.MelCodeGenerator(h)
    return g._config()


def test_create_validates_without_cuda(pkg):
    lib = pkg._cabi.load()
    cfg = _cfg(pkg)
    hnd = C.c_void_p()
    assert lib.l2s_create(C.byref(cfg), C.byref(hnd)) == pkg._cabi.OK
    assert lib.l2s_hop(hnd) == 160
    # bf16 mode: 1 speaker projection + 1 conditioning + conv_pre + 5 ups + conv_post + 18 fused ResBlock steps
    # (C = 256, 128: one launch per step) + 6 whole-ResBlock kernels (C = 64, 16) + 1 time-packed stage kernel (C = 32:
    # the three ResBlocks of the stage in one launch)
    assert lib.l2s_launch_count(hnd, 16, 400) == 33
    assert lib.l2s_debug_set(b"pk_chan", 16 | 32 | 64) == pkg._cabi.OK
    assert lib.l2s_launch_count(hnd, 16, 400) == 29     # every C <= 64 stage as one time-packed launch
    assert lib.l2s_debug_set(b"pk_fuse", 0) == pkg._cabi.OK
    assert lib.l2s_launch_count(hnd, 16, 400) == 35     # one launch per ResBlock on the C <= 64 stages
    assert lib.l2s_debug_set(b"pk_fuse", 1) == pkg._cabi.OK
    assert lib.l2s_debug_set(b"pk_chan", 32) == pkg._cabi.OK
    assert lib.l2s_debug_set(b"fuse_branch", 0) == pkg._cabi.OK
    assert lib.l2s_launch_count(hnd, 16, 400) == 53     # every ResBlock step its own launch
    assert lib.l2s_debug_set(b"fuse_branch", 1) == pkg._cabi.OK
    cfg32 = _cfg(pkg)
    cfg32.precision = pkg._cabi.PREC_FP32
    h32 = C.c_void_p()
    assert lib.l2s_create(C.byref(cfg32), C.byref(h32)) == pkg._cabi.OK
    assert lib.l2s_launch_count(h32, 16, 400) == 98      # fp32 mode: every conv is its own launch
    lib.l2s_destroy(h32)
    assert lib.l2s_workspace_bytes(hnd, 16, 400) > 0
    assert lib.l2s_workspace_bytes(hnd, 0, 400) < 0
    # forward before finalize is a state error, not a crash
    assert lib.l2s_forward(hnd, None, None, None, 0, None, 1, 1, 2, None, None, 0) == pkg._cabi.ERR_STATE
    # wrong weight name / size
    buf = (C.c_float * 4)()
    assert lib.l2s_set_weight(hnd, b"nope.weight", buf, 4) == pkg._cabi.ERR_INVALID
    assert lib.l2s_set_weight(hnd, b"conv_post.bias", buf, 4) == pkg._cabi.ERR_SHAPE
    assert b"conv_post.bias" in lib.l2s_last_error(hnd)
    lib.l2s_destroy(hnd)

    bad = _cfg(pkg)
    bad.model_in_dim = 300
    assert lib.l2s_create(C.byref(bad), C.byref(hnd)) == pkg._cabi.ERR_SHAPE
    lib.l2s_destroy(hnd)
    bad = _cfg(pkg)
    bad.up_ksizes[0] = 10      # k - u odd: the reference's padding (k-u)//2 would not give L*u samples
    assert lib.l2s_create(C.byref(bad), C.byref(hnd)) == pkg._cabi.ERR_UNSUPPORTED
    lib.l2s_destroy(hnd)


def _finalize_without_a_gpu(q):
    import sys
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    pkg = ge.load_package()
    lib = pkg._cabi.load()
    g = pkg.MelCodeGenerator(pkg.AttrDict(vo.shipped_config()))
    cfg = g._config()
    hnd = C.c_void_p()
    created = lib.l2s_create(C.byref(cfg), C.byref(hnd))
    keep, rejected = [], []
    for name, t in g._plain_weights().items():
        t = t.float().contiguous()
        keep.append(t)
        if lib.l2s_set_weight(hnd, name.encode(), t.data_ptr(), t.numel()) != 0:
            rejected.append(name)
    q.put((created, rejected, lib.l2s_finalize(hnd, 0), lib.l2s_last_error(hnd)))
    lib.l2s_destroy(hnd)


def test_finalize_fails_loudly_without_a_gpu(pkg, monkeypatch):
    """The library in a process that sees no CUDA device (CUDA_VISIBLE_DEVICES empty), so this also runs on a GPU
    machine."""
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    p = ctx.Process(target=_finalize_without_a_gpu, args=(q,))
    p.start()
    created, rejected, status, err = q.get(timeout=300)
    p.join(timeout=60)
    assert p.exitcode == 0
    assert created == pkg._cabi.OK
    assert rejected == []
    assert status == pkg._cabi.ERR_CUDA
    assert b"no CPU fallback" in err


def test_host_class_surface(pkg):
    h = vo.shipped_config()
    sd = vo.init_state_dict(h, seed=1234, style="trained")
    g = pkg.MelCodeGenerator(pkg.AttrDict(h))
    assert set(g.state_dict()) == set(sd) and len(sd) == 298
    g.load_state_dict(sd, strict=True)
    with pytest.raises(RuntimeError):
        g.load_state_dict({k: v for k, v in sd.items() if k != "fc.bias"}, strict=True)
    assert g.eval() is g
    g.remove_weight_norm()
    folded = vo.fold_weight_norm(sd)
    assert set(g.state_dict()) == set(folded) and len(folded) == 201
    for k, v in g._plain_weights().items():
        assert torch.equal(v, folded[k]), k
    with pytest.raises(ValueError):
        g.remove_weight_norm()      # torch's remove_weight_norm raises when there is nothing to remove
    # no CPU fallback
    code, mel, spkr = vo.synthetic_inputs(1, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        g(code=code, mel=mel, spkr=spkr)
    with pytest.raises(KeyError):
        g(code=code, spkr=spkr)


def test_constructor_reads_h_like_the_reference(pkg):
    h = vo.shipped_config()
    del h["text_supervision"]
    with pytest.raises(AttributeError):          # models_multi_input.py:31 reads h.text_supervision
        pkg.MelCodeGenerator(pkg.AttrDict(h))
    with pytest.raises(NotImplementedError):
        pkg.MelCodeGenerator(pkg.AttrDict(vo.shipped_config(text_supervision=True)))
    with pytest.raises(NotImplementedError):
        pkg.MelCodeGenerator(pkg.AttrDict(vo.shipped_config(resblock="2")))
    hu = vo.unit_only_config()
    gu = pkg.CodeGenerator(pkg.AttrDict(hu))
    sdu = vo.init_state_dict(hu, seed=1234, style="trained", unit_only=True)
    gu.load_state_dict(sdu, strict=True)
    assert gu._config().variant == pkg._cabi.VARIANT_UNIT_ONLY
