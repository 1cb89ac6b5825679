"""CPU: the oracle restatement against the UNMODIFIED reference's own loss, gradient and mask outputs on seeded inputs.
When the reference sources are available (`oracle/ref_loader.py`, GA_REFERENCE_ROOT) the reference is executed live;
otherwise the test reads what the same reference calls (`oracle/gen_golden.py`: gen_loss, gen_parse, gen_masks)
returned when tests/golden/reference_kat.* was written.  Either way the comparison and its tolerances are the same.
It runs in a subprocess because `oracle/ref_loader.py` neutralises `.cuda()` process-wide."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_LIVE = r'''
import json, os, sys
import numpy as np
import torch
sys.path.insert(0, %(root)r)
from oracle import ref_loader, gen_golden, oracle as O
from oracle.cases import LOSS_CASES, MASK_CASES, make_loss_inputs
from oracle.specs import tokens_from_record
live = ref_loader.available()
if live:
    ref = ref_loader.load()
    arrays = {}
    recs = gen_golden.gen_loss(ref, arrays)              # the reference's own code, right now
    parse_recs = gen_golden.gen_parse(ref)
else:                                                    # what the same calls returned when the fixtures were written
    with open(os.path.join(gen_golden.GOLDEN, "reference_kat.json")) as f:
        kat = json.load(f)
    arrays = dict(np.load(os.path.join(gen_golden.GOLDEN, "reference_kat.npz")))
    recs = [next(r for r in kat["loss"] if r["name"] == c["name"]) for c in LOSS_CASES]
    parse_recs = kat["parse"]
out = {"source": "live" if live else "stored", "loss": [], "masks": 0}
parse = {p["meta_prompt"]: p for p in parse_recs if "error" not in p}
for case, rec in zip(LOSS_CASES, recs):
    if case.get("normalize_eot") or parse[case["meta_prompt"]]["custom"]:
        continue                                          # covered by the fixture test; keep the live check small
    tokens = tokens_from_record(parse[case["meta_prompt"]])
    hp = O.HyperParams(**{k: v for k, v in (case.get("hyper") or {}).items() if k in O.HyperParams.__annotations__})
    hp.sub_prompt_avg_within = (case.get("cfg") or {}).get("sub_prompt_avg_within", False)
    Ps, _ = make_loss_inputs(case)
    for P in Ps:
        P.requires_grad_(True)
    store = {"down_cross": [], "mid_cross": [], "up_cross": []}
    for P, place in zip(Ps, case["places"]):
        store[place + "_cross"].append(P)
    r = O.guidance_loss(O.aggregate_attention(store, 16), tokens, 16, hp, smooth_attentions=case.get("smooth", True))
    row = {"name": case["name"], "ref_total": rec["total"], "oracle_total": float(r.loss)}
    if float(r.loss) != 0:
        g = torch.autograd.grad(r.loss, Ps)[0]
        n_maps = sum(P.shape[0] for P in Ps)
        mine = (g[0] * n_maps).reshape(16, 16, -1).numpy()
        gold = arrays["loss_" + case["name"] + "_dAbar"]
        row["grad_rel"] = float(np.abs(mine - gold).max() / max(np.abs(gold).max(), 1e-30))
    out["loss"].append(row)
mask_recs = gen_golden.gen_masks(ref) if live else kat["masks"]
assert len(mask_recs) == len(MASK_CASES)
for (box, res, shrink), rec in zip(MASK_CASES, mask_recs):
    assert (rec["box"], rec["res"], rec["shrink"]) == (list(box), res, shrink), rec
    m = O.inside_box_mask(O.rect_of_size(tuple(box), float(res) if res == 16 else res), res, shrink)
    assert ["".join(map(str, row)) for row in m.tolist()] == rec["mask_rows"], box
    out["masks"] += 1
print("LIVE_RESULT " + json.dumps(out))
'''


@pytest.mark.reference
def test_oracle_matches_the_reference_run_live():
    r = subprocess.run([sys.executable, "-c", _LIVE % {"root": ROOT}], capture_output=True, text=True, timeout=600,
                       cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = next(l for l in r.stdout.splitlines() if l.startswith("LIVE_RESULT "))
    out = json.loads(line[len("LIVE_RESULT "):])
    assert out["masks"] > 0 and len(out["loss"]) >= 6
    for row in out["loss"]:
        assert row["oracle_total"] == pytest.approx(row["ref_total"], rel=1e-5), row
        if "grad_rel" in row:
            assert row["grad_rel"] < 1e-4, row
