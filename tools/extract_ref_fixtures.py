#!/usr/bin/env python
"""Extract the reference's own test fixtures (data only) into tests/golden/.

Runs in the dev container (needs /root/reference). Outputs are committed:
  tests/golden/state_test_logs.json — the inline mjai JSON logs of libriichi/src/state/test.rs,
      keyed by test fn name, in source order (assert logic is re-stated in tests/test_oracle_state.py)
  tests/golden/golden_game.jsonl — the seeded full-game log embedded in log-viewer/index.example.html:10-264
  tests/golden/ref_tables.json — libriichi's shanten / agari data files (algo/data/*.bin.gz) as a digest of their whole
      content plus a seeded sample of rows / keys (tests/test_tables.py compares the generated tables against both)
  tests/golden/ref_model_outputs.json — for network versions 2-4 at 32 channels x 2 blocks: the key schema of mortal/model.py's
      Brain / DQN state_dicts, the seeds of tests/ref_checkpoint_fixture.py's weights and inputs, and the Q-values Mortal's
      modules compute from them (fp32, CPU); tests/test_reference_checkpoint.py loads the same weights into mortal_b200
"""
import gzip
import hashlib
import json
import os
import re
import sys

import numpy as np

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def agari_digest(table: dict) -> str:
    """sha256 of a key -> ordered div list map, independent of the record order of the file it came from"""
    text = "".join(f"{k:x}:{','.join(str(d) for d in table[k])}\n" for k in sorted(table))
    return hashlib.sha256(text.encode()).hexdigest()


def table_fixtures() -> dict:
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import gen_agari_table

    data = os.path.join(REF, "libriichi/src/algo/data")
    rng = np.random.default_rng(2024)
    out = {}
    for name, n_sample in (("shanten_suhai.bin", 512), ("shanten_jihai.bin", 256)):
        with gzip.open(os.path.join(data, name + ".gz"), "rb") as f:
            raw = f.read()
        rows = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 5)
        idx = np.sort(rng.choice(rows.shape[0], n_sample, replace=False))
        out[name] = {"bytes": len(raw), "sha256": hashlib.sha256(raw).hexdigest(),
                     "sample_rows": {str(int(i)): rows[i].tobytes().hex() for i in idx}}
    with gzip.open(os.path.join(data, "agari.bin.gz"), "rb") as f:
        table = gen_agari_table.parse(f.read())
    keys = sorted(table)
    pick = np.sort(rng.choice(len(keys), 256, replace=False))
    out["agari.bin"] = {"keys": len(table), "sha256": agari_digest(table),
                        "sample": {f"{keys[i]:x}": table[keys[i]] for i in pick}}
    return out


def model_fixtures() -> dict:
    """Mortal's own Brain / DQN (mortal/model.py) on seeded weights and inputs, fp32 on the CPU: the key schema of each
    version's state_dicts and the Q-values for tests/ref_checkpoint_fixture.py's inputs. Data only."""
    import importlib.util
    import types

    import torch

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import ref_checkpoint_fixture as F
    from mortal_b200.libriichi import consts

    # mortal/model.py imports only obs_shape / oracle_obs_shape / ACTION_SPACE / GRP_SIZE from libriichi.consts
    pkg = types.ModuleType("libriichi")
    pkg.consts = consts
    sys.modules.setdefault("libriichi", pkg)
    sys.modules.setdefault("libriichi.consts", consts)
    spec = importlib.util.spec_from_file_location("mortal_reference_model", os.path.join(REF, "mortal/model.py"))
    model = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(model)
    torch.set_num_threads(4)
    out = {"channels": F.CHANNELS, "blocks": F.BLOCKS, "rows": F.ROWS, "versions": {}}
    for version in F.VERSIONS:
        brain = model.Brain(conv_channels=F.CHANNELS, num_blocks=F.BLOCKS, version=version)
        dqn = model.DQN(version=version)
        strip = lambda sd: {k: tuple(v.shape) for k, v in sd.items() if not k.endswith("num_batches_tracked")}
        schema = (strip(brain.state_dict()), strip(dqn.state_dict()))
        weight_seed, input_seed = 7000 + version, 8000 + version
        bsd, dsd = F.make_state_dicts(schema, weight_seed)
        brain.load_state_dict({k: torch.from_numpy(v) for k, v in bsd.items()}, strict=False)
        dqn.load_state_dict({k: torch.from_numpy(v) for k, v in dsd.items()})
        brain.eval(), dqn.eval()
        obs, masks = F.make_inputs(version, F.ROWS, input_seed)
        with torch.no_grad():
            q = dqn(brain(torch.from_numpy(obs)), torch.from_numpy(masks)).double().numpy()
        out["versions"][str(version)] = {
            "brain_schema": [[k, list(s)] for k, s in schema[0].items()],
            "dqn_schema": [[k, list(s)] for k, s in schema[1].items()],
            "weight_seed": weight_seed, "input_seed": input_seed,
            "q": [[None if np.isneginf(x) else float(x) for x in row] for row in q],
        }
    return out


def main():
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "ref_model_outputs.json"), "w") as f:
        json.dump(model_fixtures(), f)
        f.write("\n")
    src = open(os.path.join(REF, "libriichi/src/state/test.rs")).read()
    logs = {}
    cur = None
    for m in re.finditer(r'fn (\w+)\(\)|r#"(.*?)"#', src, re.S):
        if m.group(1):
            cur = m.group(1)
            continue
        body = m.group(2)
        lines = [ln.strip() for ln in body.strip().split("\n") if ln.strip()]
        for ln in lines:
            json.loads(ln)
        logs.setdefault(cur, []).append(lines)
    with open(os.path.join(OUT, "state_test_logs.json"), "w") as f:
        json.dump(logs, f, indent=0)
    print({k: [len(x) for x in v] for k, v in logs.items()})

    html = open(os.path.join(REF, "log-viewer/index.example.html")).read()
    m = re.search(r"allActions = `\n(.*?)\n\s*`", html, re.S)
    lines = [ln for ln in m.group(1).split("\n") if ln.strip()]
    for ln in lines:
        json.loads(ln)
    with open(os.path.join(OUT, "golden_game.jsonl"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("golden game lines:", len(lines))

    with open(os.path.join(OUT, "ref_tables.json"), "w") as f:
        json.dump(table_fixtures(), f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
