"""The committed golden vectors are what the UNMODIFIED reference produces: given a checkout of the original rl4mm project
(the environment variable RL4MM_REFERENCE), part of them is regenerated through oracle/refshim.py -- in a subprocess,
because the shims put stub modules into sys.modules -- and compared with the files in tests/golden/.  The reference is not
part of this repository, so without RL4MM_REFERENCE the test is skipped; every other test reads the committed vectors."""
import os
import subprocess
import sys
from pathlib import Path

import pytest

REFERENCE = os.environ.get("RL4MM_REFERENCE")
ROOT = Path(__file__).resolve().parent.parent
pytestmark = pytest.mark.skipif(not REFERENCE, reason="needs RL4MM_REFERENCE, a checkout of the original rl4mm project")

SCRIPT = r"""
import contextlib, gzip, io, json, sys, warnings
from pathlib import Path
root, tmp, fn_name, file_name = Path(sys.argv[1]), Path(sys.argv[2]), sys.argv[3], sys.argv[4]
sys.path.insert(0, str(root))
from oracle import gen_golden, refshim
refshim.install()
gen_golden.GOLDEN = tmp
with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
    warnings.simplefilter("ignore")
    getattr(gen_golden, fn_name)()
new = json.loads(gzip.open(tmp / file_name).read())
old = json.loads(gzip.open(root / "tests" / "golden" / file_name).read())
sys.exit(0 if json.dumps(new, sort_keys=True) == json.dumps(old, sort_keys=True) else 3)
"""


@pytest.mark.parametrize("fn_name,file_name", [("golden_beta_ladders", "beta_ladders.json.gz"),
                                               ("golden_episode_summary", "episode_summary.json.gz"),
                                               ("golden_fixture_replay", "fixture_replay.json.gz"),
                                               ("golden_generator_merge", "generator_merge.json.gz"),
                                               ("golden_rolling_sharpe_1e12", "rolling_sharpe_1e12.json.gz"),
                                               ("golden_episode_starts", "episode_starts.json.gz")])
def test_goldens_regenerate_identically(fn_name, file_name, tmp_path):
    res = subprocess.run([sys.executable, "-c", SCRIPT, str(ROOT), str(tmp_path), fn_name, file_name], capture_output=True, text=True,
                         timeout=600)
    assert res.returncode == 0, (res.returncode, res.stderr[-2000:])
