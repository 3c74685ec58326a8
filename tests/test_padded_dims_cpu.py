"""Layout of a model whose dims are not multiples of 64 (rvae_param_layout_padded); no GPU needed."""
import ctypes

import pytest

from rawaudiovae_kelsey_b200 import _lib, engine


def _padded(S, H, L):
    lib = _lib.load()
    lay, sp, hp, lp = _lib.Layout(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    rc = lib.rvae_param_layout_padded(S, H, L, ctypes.byref(lay), ctypes.byref(sp), ctypes.byref(hp), ctypes.byref(lp))
    return rc, lay, sp.value, hp.value, lp.value


FIELDS = ("w1", "w2", "w3", "w4", "b1", "b2", "b3", "b4", "total")


@pytest.mark.parametrize("dims", [(1024, 2048, 256), (4096, 4096, 256), (64, 64, 64), (1024, 2048, 64)])
def test_padded_layout_equals_layout_for_multiples_of_64(dims):
    lib = _lib.load()
    ref = _lib.Layout()
    assert lib.rvae_param_layout(*dims, ctypes.byref(ref)) == 0
    rc, lay, sp, hp, lp = _padded(*dims)
    assert rc == 0 and (sp, hp, lp) == dims
    assert all(getattr(lay, f) == getattr(ref, f) for f in FIELDS)
    # parameters are contiguous and where they were before
    geo = engine.param_geometry(*dims)
    S, H, L = dims
    assert geo["fc22.weight"][0] == lay.w2 + L * H
    for name, (off, shape, strides) in geo.items():
        assert strides == (shape[1], 1) if len(shape) == 2 else strides == (1,), name
    assert engine.param_offsets(*dims) == {n: (o, sh) for n, (o, sh, _) in geo.items()}


@pytest.mark.parametrize("dims,pads", [((1000, 300, 16), (1024, 320, 64)), ((250, 100, 3), (256, 128, 64)),
                                       ((1, 1, 1), (64, 64, 64)), ((1024, 2000, 16), (1024, 2048, 64)),
                                       ((65, 64, 129), (128, 64, 192))])
def test_padded_offsets(dims, pads):
    S, H, L = dims
    rc, lay, sp, hp, lp = _padded(S, H, L)
    assert rc == 0 and (sp, hp, lp) == pads
    o = 0
    for f, n in (("w1", hp * sp), ("w2", 2 * lp * hp), ("w3", hp * lp), ("w4", sp * hp), ("b1", hp), ("b2", 2 * lp),
                 ("b3", hp), ("b4", sp)):
        assert getattr(lay, f) == o, f
        o += n
    assert lay.total == o
    # rvae_param_layout keeps rejecting other dims
    assert _lib.load().rvae_param_layout(S, H, L, ctypes.byref(_lib.Layout())) == (0 if dims == pads else 2)


@pytest.mark.parametrize("dims", [(1000, 300, 16), (250, 100, 3), (1024, 2000, 16)])
def test_parameter_geometry_agrees_with_layout(dims):
    S, H, L = dims
    rc, lay, sp, hp, lp = _padded(S, H, L)
    geo = engine.param_geometry(S, H, L)
    assert geo == {
        "fc1.weight": (lay.w1, (H, S), (sp, 1)), "fc1.bias": (lay.b1, (H,), (1,)),
        "fc21.weight": (lay.w2, (L, H), (hp, 1)), "fc21.bias": (lay.b2, (L,), (1,)),
        "fc22.weight": (lay.w2 + lp * hp, (L, H), (hp, 1)), "fc22.bias": (lay.b2 + lp, (L,), (1,)),
        "fc3.weight": (lay.w3, (H, L), (lp, 1)), "fc3.bias": (lay.b3, (H,), (1,)),
        "fc4.weight": (lay.w4, (S, H), (hp, 1)), "fc4.bias": (lay.b4, (S,), (1,)),
    }
    # every parameter lies inside its block, and no two parameters share an element
    blocks = {"fc1.weight": ("w1", hp * sp), "fc21.weight": ("w2", 2 * lp * hp), "fc22.weight": ("w2", 2 * lp * hp),
              "fc3.weight": ("w3", hp * lp), "fc4.weight": ("w4", sp * hp), "fc1.bias": ("b1", hp),
              "fc21.bias": ("b2", 2 * lp), "fc22.bias": ("b2", 2 * lp), "fc3.bias": ("b3", hp), "fc4.bias": ("b4", sp)}
    seen = set()
    for name, (off, shape, strides) in geo.items():
        start = getattr(lay, blocks[name][0])
        rows, cols = (shape[0], shape[1]) if len(shape) == 2 else (1, shape[0])
        pitch = strides[0] if len(shape) == 2 else cols
        idx = {off + r * pitch + c for r in range(rows) for c in range(cols)}
        assert min(idx) >= start and max(idx) < start + blocks[name][1], name
        assert not (idx & seen), name
        seen |= idx


def test_padded_layout_rejects_bad_dims():
    for dims in [(0, 64, 64), (64, -1, 64), (64, 64, 0)]:
        assert _padded(*dims)[0] == 2
