"""Generates tests/golden/reference_signatures.json from a checkout of the reference (the directory that holds RL-SHEMS/):
what tests/test_julia_shim_static.py needs to know about the REFERENCE's Julia sources — function signatures of algorithms/DDPG.jl and
src/memory_plotting_saving.jl, how the kept memory functions touch the global `memory`, the calls and includes of
DDPG_reinforce_charger_v1.jl and the globals assigned by input.jl / DDPG.jl / the driver.  Facts (names and arities), not code.
    python tests/golden/make_reference_signatures.py <reference checkout>"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import test_julia_shim_static as T  # noqa: E402

if __name__ == "__main__":
    facts = T.reference_facts(sys.argv[1])
    with open(os.path.join(HERE, "reference_signatures.json"), "w") as f:
        json.dump(facts, f, indent=1, ensure_ascii=False, sort_keys=True)
    print({k: len(v) for k, v in facts.items()})
