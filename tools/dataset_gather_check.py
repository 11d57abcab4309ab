"""selfplay.gather_dataset under torchrun (each rank records its own block of game ids on its own GPU, rank 0 gathers them) against
one engine on rank 0's GPU recording every game alone:
     torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29515 tools/dataset_gather_check.py
Rank 0 compares the two datasets record for record in canonical order (features, meta, origin, each record's options and regrets;
a gathered record's tree is its game's index in its own rank's call), then trains on both from the same model and seed and
compares the losses and the final weights bit for bit.  Prints one JSON line on rank 0."""
import json
import os
import sys
import tempfile
import time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
from citadels_self_play_b200 import Engine, arena, selfplay
from citadels_self_play_b200.value_model import ValueOnlyNN

N, SEED, GID0 = 24, 20261020, 90_000
seats = [arena.deep(20, 10, 5.0), arena.pure(40), arena.random_seat(), arena.pure(30), arena.random_seat(), arena.deep(20, 10, 5.0)]
torch.manual_seed(1)
model = ValueOnlyNN(418, 512).eval()
ROOM = 100_000
eng = Engine(capacity=64, device=local)
rec = selfplay.record_arena(N, seats, record_seats=[0, 1, 3, 5], models=[model], mode="tree", threshold=2.0, engine=eng, seed=SEED,
                            first_gid=GID0, max_records=ROOM * (world if rank == 0 else 1))
dist.barrier()
t0 = time.perf_counter()
counts = selfplay.gather_dataset(eng, dst=0)
gather_s = time.perf_counter() - t0
if rank == 0:
    solo = Engine(capacity=64, device=local)
    solo.set_value_model(model)
    solo.dataset_reserve(ROOM * world, 16 * ROOM * world)
    solo.arena(N, seats, seed=SEED, first_gid=GID0, record=([0, 1, 3, 5], selfplay.MODES["tree"], 2.0))
    g, s = eng.dataset_read(), solo.dataset_read()
    n = len(s["meta"])
    assert n > 0 and len(g["meta"]) == n and sum(counts["records"]) == n, (len(g["meta"]), n, counts)
    assert g["origin"].tobytes() == s["origin"].tobytes()
    assert g["features"].tobytes() == s["features"].tobytes()
    firsts = [arena.rank_block(N, r, world)[0] for r in range(world)]
    for i in range(n):
        a, b = g["meta"][i], s["meta"][i]
        for k in ("node", "n_options", "seat", "role_pick"):
            assert int(a[k]) == int(b[k]), (i, k)
        assert a["node_value"].tobytes() == b["node_value"].tobytes(), i
        game = int(s["origin"][i]["gid"]) - GID0
        block = max(r for r in range(world) if firsts[r] <= game)
        assert int(a["tree"]) == int(b["tree"]) - firsts[block], i
        oa, ob, k = int(a["option_offset"]), int(b["option_offset"]), int(a["n_options"])
        assert g["options"][oa:oa + k].tobytes() == s["options"][ob:ob + k].tobytes(), i
        assert g["regrets"][oa:oa + k].tobytes() == s["regrets"][ob:ob + k].tobytes(), i
    trained = []
    with tempfile.TemporaryDirectory(prefix="gather_check_") as tmp:
        for e, name in ((eng, "gathered"), (solo, "solo")):
            d = e.dataset_read()
            tr, va = selfplay.split_by_game(d["origin"], 0.2, seed=3, rows=d["row"])
            torch.manual_seed(5)
            h = {}
            best = selfplay.train_on_dataset(e, tr, va, "node_value", epochs=3, lr=1e-3, batch_size=32, model=ValueOnlyNN(418, 512),
                                             seed=9, parent_folder=os.path.join(tmp, name), history=h)
            trained.append((best, h))
    (ba, ha), (bb, hb) = trained
    assert ba == bb and ha["train_losses"] == hb["train_losses"] and ha["eval_losses"] == hb["eval_losses"]
    for k, v in hb["final_state"].items():
        assert np.array_equal(ha["final_state"][k], v), k
    solo.close()
    print(json.dumps(dict(world=world, games=N, records=n, rank_records=counts["records"], gather_s=gather_s,
                          gpu=torch.cuda.get_device_name(local), equals_single_engine=True, training_bit_identical=True)), flush=True)
eng.close()
dist.barrier()
dist.destroy_process_group()
