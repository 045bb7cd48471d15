"""CPU tests of the N>1 plumbing (gloo, world_size 2) and of bench.py's JSON contract for the reference arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

from conftest import ROOT


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from katago_b200 import modelgen
    from katago_b200.dist_weights import broadcast_model_bytes, shard_games
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    data = modelgen.model_bytes("tiny_nbt", seed=9) if rank == 0 else None
    got = broadcast_model_bytes(data, 0)
    games = shard_games(10, rank, world)
    with open(os.path.join(out_dir, f"r{rank}.json"), "w") as f:
        import hashlib
        json.dump({"sha": hashlib.sha256(got).hexdigest(), "n": len(got), "games": games}, f)
    dist.barrier()
    dist.destroy_process_group()


def test_weight_broadcast_and_game_sharding_world2(tmp_path):
    import hashlib
    from katago_b200 import modelgen
    port = 29500 + os.getpid() % 2000
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    expect = hashlib.sha256(modelgen.model_bytes("tiny_nbt", seed=9)).hexdigest()
    r = [json.load(open(tmp_path / f"r{i}.json")) for i in range(2)]
    assert r[0]["sha"] == r[1]["sha"] == expect
    assert sorted(r[0]["games"] + r[1]["games"]) == list(range(10)) and not set(r[0]["games"]) & set(r[1]["games"])


class _RecordingHandle:
    """Stands in for nn_backend.ComputeHandle (no GPU here): records what WeightBroadcaster asks of it."""
    def __init__(self):
        self.calls = []
    def comm_init(self, uid, rank, world): self.calls.append(("comm_init", uid, rank, world))
    def stage_weights(self, m): self.calls.append(("stage", m))
    def wait_staged(self): self.calls.append(("wait_staged",))
    def broadcast_staged_weights(self, root): self.calls.append(("bcast", root)); return 1.5
    def commit_weights(self): self.calls.append(("commit",))


def _wb_worker(rank, world, port, tmp):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from katago_b200.dist_weights import WeightBroadcaster
    h = _RecordingHandle()
    wb = WeightBroadcaster(h, src=0, id_source=lambda: bytes(range(128)))
    ms = wb.update("net-A" if rank == 0 else None)
    with open(os.path.join(tmp, f"wb{rank}.json"), "w") as f:
        json.dump({"calls": [[c[0]] + [x if not isinstance(x, bytes) else list(x) for x in c[1:]] for c in h.calls], "ms": ms}, f)
    dist.barrier()
    dist.destroy_process_group()


def test_weight_broadcaster_world2_protocol(tmp_path):
    """Every rank joins the communicator with the source's id; only the source stages; all broadcast, then commit."""
    port = 31500 + os.getpid() % 2000
    mp.spawn(_wb_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r = [json.load(open(tmp_path / f"wb{i}.json")) for i in range(2)]
    uid = list(range(128))
    assert r[0]["calls"] == [["comm_init", uid, 0, 2], ["stage", "net-A"], ["wait_staged"], ["bcast", 0], ["commit"]]
    assert r[1]["calls"] == [["comm_init", uid, 1, 2], ["bcast", 0], ["commit"]]
    assert r[0]["ms"] == r[1]["ms"] == 1.5


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "kgref_cpu_selfplay")),
                    reason="the reference arm runs oracle/_ref/kgref_cpu_selfplay, built only where the reference's sources are")
def test_bench_reference_arm_prints_contract_json():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny_nbt", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    for k in ("metric", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config"):
        assert k in d
