"""bench.py --dump-outputs: the saved arrays are the tables and the loss after exactly warmup + steps training steps on
the benchmark's seeded inputs, replayed here through KGEEngine."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    steps, warmup = 3, 2
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--no-extra", "--no-cpu", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    got = {n: np.load(tmp_path / (n + ".npy")) for n in ("ent_embeddings", "rel_embeddings", "last_step_loss")}
    assert sorted(os.listdir(tmp_path)) == sorted(n + ".npy" for n in got)
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20

    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    from ampligraph_b200.engine import KGEEngine
    from ampligraph_b200.parallel import batch_slot, tables_close
    c, B = bench.CFG, bench.CFG["batch"]
    rng = np.random.default_rng(0)
    K = bench.internal_k(c)
    ent0, rel0 = bench.glorot(c["n_ent"], K, rng), bench.glorot(c["n_rel"], K, rng)
    data = bench.synthetic_kg(c["n_ent"], c["n_rel"], c["n_triples"])
    eng = KGEEngine(c["model"], c["k"], c["eta"], c["n_ent"], c["n_rel"], loss=c["loss"], loss_params=c["loss_params"],
                    optimizer=c["optimizer"], optimizer_params={"learning_rate": c["lr"]})
    eng.set_embeddings(ent0, rel0)
    eng.set_hot_entities(triples=data)
    dev, nb = torch.as_tensor(data).cuda(), len(data) // B
    for i in range(warmup + steps):
        if i == warmup + steps - 1:
            eng.read_loss()  # keep only the last step's loss
        j = batch_slot(i, 1, 0, nb)
        eng.train_step(dev[j * B:(j + 1) * B], None, seed=1234, step=i)
    loss = eng.loss_acc.cpu().numpy()
    ent, rel = (x.cpu().numpy() for x in eng.get_embeddings())
    eng.close()
    assert got["ent_embeddings"].shape == ent.shape and got["rel_embeddings"].shape == rel.shape
    # one Adam step more or less moves every touched parameter by about lr: far outside tables_close
    assert tables_close(got["ent_embeddings"], ent, ent0)[0] and tables_close(got["rel_embeddings"], rel, rel0)[0]
    assert got["last_step_loss"].shape == (2,) and np.allclose(got["last_step_loss"], loss, rtol=1e-5), (got["last_step_loss"], loss)
