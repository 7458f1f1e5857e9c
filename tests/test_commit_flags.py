"""ptc_scene_commit_ex flags through the Python wrapper (no device needed)."""
import pytest


def _scene(pt):
    s = pt.Scene()
    m = s.add_material(pt.lambertian((1, 1, 1)))
    s.add_mesh([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.5]], [[0, 1, 2], [1, 3, 2]], m)
    return s


@pytest.mark.parametrize("kw, flags", [({}, 0), ({"fast_build": True}, 1), ({"device_sah": True}, 2)])
def test_commit_passes_flags(pt, monkeypatch, kw, flags):
    assert (pt.COMMIT_FAST_BUILD, pt.COMMIT_DEVICE_SAH) == (1, 2)
    seen = []
    monkeypatch.setattr(pt.core(), "ptc_scene_commit_ex", lambda h, device, f: seen.append((device, f)) or 0)
    _scene(pt).to_core().commit(0, **kw)
    assert seen == [(0, flags)]


def test_device_sah_commit_without_device(pt):
    if pt.device_count() > 0:
        pytest.skip("a CUDA device is present")
    cs = _scene(pt).to_core()
    with pytest.raises(pt.PtcError) as e:
        cs.commit(0, device_sah=True)
    assert e.value.code == pt.PTC_E_CUDA
    with pytest.raises(pt.PtcError) as e:
        cs.commit(0, fast_build=True, device_sah=True)  # arguments are checked before the device is looked for
    assert e.value.code == pt.PTC_E_INVALID
