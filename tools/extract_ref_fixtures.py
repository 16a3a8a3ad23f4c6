#!/usr/bin/env python
"""Extract the reference's own test fixtures (data only) into tests/golden/.

Runs in the dev container (needs /root/reference). Outputs are committed:
  tests/golden/state_test_logs.json — the inline mjai JSON logs of libriichi/src/state/test.rs,
      keyed by test fn name, in source order (assert logic is re-stated in tests/test_oracle_state.py)
  tests/golden/golden_game.jsonl — the seeded full-game log embedded in log-viewer/index.example.html:10-264
  tests/golden/ref_tables.json — libriichi's shanten / agari data files (algo/data/*.bin.gz) as a digest of their whole
      content plus a seeded sample of rows / keys (tests/test_tables.py compares the generated tables against both)
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


def main():
    os.makedirs(OUT, exist_ok=True)
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
