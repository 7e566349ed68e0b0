"""ORACLE / TEST INFRASTRUCTURE — not part of the shipped product.

Golden table of the labeler's instruction strings (arp_dt/data_procgen.py:281-317, arp_dt/assets/procgen_instruct.py:
72-105): get_clip_instruct(env) for every env of ENVS, get_clip_special_instruct(env, inst) for every pair of ENVS x
INSTS (a pair the function refuses is stored as RAISES), and the positive / negative prompt lists of
PROCGEN_POS_NEG_INSTRUCT for the envs arp_b200.instructions.POS_NEG restates. Writes tests/golden/instructions.json.

  python -m oracle.make_golden_instructions                  # from the REFERENCE's own functions (needs the reference)
  python -m oracle.make_golden_instructions --restatement    # from arp_b200/instructions.py, where no reference exists
"""
from __future__ import annotations

import importlib
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle import stubs  # noqa: E402

GOLDEN = ROOT / "tests" / "golden" / "instructions.json"
ENVS = ("coinrun", "coinrun_aisc", "maze", "maze_aisc", "maze_yellowline", "maze_redline_yellowgem", "x")
INSTS = ("random1", "random2", "misinfo", "misinfo2", "misinfo3", "misinfo4", "zzz")
RAISES = "raises ValueError"


def table(get_clip_instruct, get_clip_special_instruct, pos_neg: dict, pos_neg_keys) -> dict:
    special = {}
    for env in ENVS:
        special[env] = {}
        for inst in INSTS:
            try:
                special[env][inst] = get_clip_special_instruct(env, inst)
            except ValueError:
                special[env][inst] = RAISES
    return {"clip_instruct": {env: get_clip_instruct(env) for env in ENVS}, "clip_special_instruct": special,
            "pos_neg": {k: list(pos_neg[k]) for k in pos_neg_keys}}


def reference_table() -> dict:
    from arp_b200 import instructions
    stubs.import_reference()
    dp = importlib.import_module("arp_dt.data_procgen")
    pn = importlib.import_module("arp_dt.assets.procgen_instruct").PROCGEN_POS_NEG_INSTRUCT
    return table(dp.get_clip_instruct, dp.get_clip_special_instruct, pn, sorted(instructions.POS_NEG))


def restatement_table() -> dict:
    from arp_b200 import instructions
    return table(instructions.get_clip_instruct, instructions.get_clip_special_instruct, instructions.POS_NEG,
                 sorted(instructions.POS_NEG))


if __name__ == "__main__":
    if "--restatement" in sys.argv:
        source = ("arp_b200/instructions.py, the restatement that was written and committed together with the live "
                  "comparison tests/test_host_logic.py::test_instruction_strings_equal_reference and is unchanged "
                  "since; the reference was not available to run. That test checks this table against the reference "
                  "wherever the reference is present.")
        t = restatement_table()
    else:
        if not stubs.reference_available():
            sys.exit("needs the reference project (oracle/stubs.py REFERENCE); --restatement writes the table from "
                     "arp_b200/instructions.py instead")
        source = "the reference's own get_clip_instruct / get_clip_special_instruct / PROCGEN_POS_NEG_INSTRUCT"
        t = reference_table()
    GOLDEN.write_text(json.dumps({"source": source, **t}, indent=1) + "\n")
    print(f"wrote {GOLDEN.relative_to(ROOT)}: {len(ENVS)} envs x {len(INSTS)} instruction types, "
          f"{len(t['pos_neg'])} pos/neg lists")
