"""CPU: host logic of the deterministic mode.  The library exports v2s_set_deterministic; with it off the workspace size
is the default one, with it on the size grows by the mode's scratch; the Python workspace caches and the CUDA-graph key
follow torch.are_deterministic_algorithms_enabled()."""
import pytest
import torch


@pytest.fixture
def lib():
    from vit2spn import _lib
    yield _lib.lib
    _lib.lib.v2s_set_deterministic(int(torch.are_deterministic_algorithms_enabled()))


def test_switch_is_exported(lib):
    import vit2spn
    assert "v2s_set_deterministic" in vit2spn.EXPORTED
    assert lib.v2s_set_deterministic(1) == 0
    assert lib.v2s_set_deterministic(0) == 0


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_workspace_bytes_off_unchanged_on_grows(lib, mode):
    lib.v2s_set_deterministic(0)
    off = [lib.v2s_workspace_bytes(b, mode, g, s) for b in (1, 128) for g, s in ((4, 2), (1, 1), (1, 0))]
    lib.v2s_set_deterministic(1)
    on = [lib.v2s_workspace_bytes(b, mode, g, s) for b in (1, 128) for g, s in ((4, 2), (1, 1), (1, 0))]
    lib.v2s_set_deterministic(0)
    assert [lib.v2s_workspace_bytes(b, mode, g, s) for b in (1, 128) for g, s in ((4, 2), (1, 1), (1, 0))] == off
    for i, (a, b) in enumerate(zip(off, on)):
        if i % 3 == 2:
            assert a == b                   # nothing saved, no backward: no scratch
        else:
            assert b > a and (b - a) % 1024 == 0


def test_workspace_keys_follow_torch_flag(lib, monkeypatch):
    from vit2spn import modules
    sized = []
    monkeypatch.setattr(modules, "lib", type("L", (), {
        "v2s_set_deterministic": staticmethod(lambda on: sized.append(("set", on)) or 0),
        "v2s_workspace_bytes": staticmethod(lambda *a: 4096 if sized[-1] == ("set", 1) else 2048),
    }))
    monkeypatch.setattr(modules, "_workspaces", {})
    for flag, nbytes in ((False, 2048), (True, 4096), (False, 2048)):
        monkeypatch.setattr(torch, "are_deterministic_algorithms_enabled", lambda f=flag: f)
        ws = modules._scratch_workspace(torch.device("cpu"), 2, 1, 1, 0)
        assert ws.numel() == nbytes + 1024
        assert modules._new_workspace(torch.device("cpu"), 2, 1, 1, 1).numel() == nbytes + 1024
    assert set(k[-1] for k in modules._workspaces) == {False, True}
    net = modules.DualStreamNetwork.__new__(modules.DualStreamNetwork)
    net.__dict__.update(_ws={}, _ws_busy=set())
    for flag in (False, True):
        monkeypatch.setattr(torch, "are_deterministic_algorithms_enabled", lambda f=flag: f)
        net._release_workspace(net._take_workspace(torch.device("cpu"), 2, 1))
    assert sorted(k[-1] for k in net._ws) == [False, True]


def test_graph_key_follows_torch_flag():
    import inspect
    from vit2spn import modules
    src = inspect.getsource(modules.DualStreamNetwork.ssp_step_graphed)
    key = src[src.index("key = ("):src.index("graphs = ")]
    assert "torch.are_deterministic_algorithms_enabled()" in key
