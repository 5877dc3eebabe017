"""Writes tests/golden/live_digests.json: SHA-256 digests of the oracle's outputs on every case of the `test_live_*` tests
of tests/test_reference_spirv.py, which those tests check where the reference's compiled modules cannot be run.

Each test is run once per parameter set with recording on.  Where oracle/_ref/libspvref.so can be run, the same run also
asserts that the oracle equals the modules, so a digest is only written for outputs the modules reproduce.
    python tests/golden/make_live_digests.py
"""
import itertools
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import spirv_cases as cases  # noqa: E402
import test_reference_spirv as t  # noqa: E402

t.RECORD = {}
fixtures = {"ggx_lut": cases.lut_rgba8()}
for name in sorted(n for n in dir(t) if n.startswith("test_live_")):
    fn = getattr(t, name)
    marks = [m for m in getattr(fn, "pytestmark", []) if m.name == "parametrize"]
    axes = [([m.args[0]] if "," not in m.args[0] else m.args[0].split(","), m.args[1]) for m in marks]
    for combo in itertools.product(*[values for _, values in axes]):
        kwargs = dict(fixtures) if "ggx_lut" in fn.__code__.co_varnames[:fn.__code__.co_argcount] else {}
        for (names, _), value in zip(axes, combo):
            kwargs.update(zip(names, value if len(names) > 1 else (value,)))
        fn(**kwargs)
        print(name, combo, flush=True)

out = {"source": "the oracle, checked equal to the reference's modules in the same run" if t.LIVE else
       "the oracle; the reference's modules were not run",
       "digests": dict(sorted(t.RECORD.items()))}
with open(t.LIVE_DIGESTS, "w") as f:
    json.dump(out, f, indent=1)
    f.write("\n")
print(len(t.RECORD), "digests ->", t.LIVE_DIGESTS)
