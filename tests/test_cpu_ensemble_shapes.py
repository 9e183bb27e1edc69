"""CPU tests of ensembles over rooms of different sizes and numbers of target sets: construction and wave planning
touch no GPU, and every member's device byte count follows its own grid, dt and number of target sets."""
import json
import os

from conftest import REPO


def test_mixed_room_ensemble_plans_per_member_bytes_without_cuda(monkeypatch):
    import torch
    from optimal_crowds_b200 import _lib, ensemble, synthetic
    monkeypatch.chdir(REPO)
    odd = synthetic.ensemble_room(n=97, agents=12)
    rooms = ["room_test", "exit_opposite", "metro_station", "slalom", odd, "metro_station"]
    configs = [{}, {"dt": 0.01}, {}, {}, {"dt": 0.025}, {"dt": 0.04}]
    for storage in ("phi", "velocity"):
        e = ensemble.ensemble(rooms, 2.0, list(range(6)), configs=configs, field_storage=storage)
        got = e.member_bytes()
        want = []
        for room, ov in zip(rooms, configs):
            if isinstance(room, str):
                with open(os.path.join(REPO, "rooms", room + ".json")) as f:
                    room = json.load(f)
            Ny, Nx = _lib.grid_shape(room["room_length"], room["room_height"], 0.05)
            keys = {" or ".join(b[5:]) for b in room["initial_boxes"].values()}
            want.append(ensemble.field_bytes_per_member(Ny, Nx, 2.0, ov.get("dt", 0.02), len(keys), storage))
        assert got == want
    # the shapes really differ: 120 x 200, 200 x 240, 160 x 320 and an odd 97 x 97; 1, 2 and 4 target sets
    assert len(set(got)) == 6
    assert ensemble.field_bytes_per_member(97, 97, 2.0, 0.02, 4) == 4 * ensemble.field_bytes_per_member(97, 97, 2.0, 0.02)
    assert not torch.cuda.is_initialized()
