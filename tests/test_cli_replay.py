"""The `mcmc` command line replays the chosen chains once for every --select output: asked for together, the outputs are the
bytes and summary lines of the runs that ask for each alone, whichever store the shared replay reads them from."""
import os
import subprocess

import pytest

from conftest import load_hex_dataset

# the lines after the throughput line, in the order they are printed
HEADS = ("selection:", "E[c]", "rank diagnostics:", "diagnostics:", "taxon pairs:", "cd marginals:", "marginals:")


@pytest.fixture(scope="module")
def S():
    import seriation_b200 as S
    if not os.path.exists(S.LIB_PATH):
        S.build()
    S.lib()
    return S


def _outputs(d):
    """flag -> (its arguments writing under directory d, the files they write)"""
    j = lambda name: str(d / name)
    return {
        "--po": (["--po", j("po.csv")], [j("po.csv")]),
        "--rank-diagnostics": (["--rank-diagnostics", j("r.csv")], [j("r.csv")]),
        "--diagnostics": (["--diagnostics", j("d.csv")], [j("d.csv")]),
        "--taxon-pairs": (["--taxon-pairs", j("T")], [j("T.%s.csv" % q) for q in ("first", "last", "precedes", "coexist")]),
        "--cd-marginals": (["--cd-marginals", j("cd.csv")], [j("cd.csv")]),
        "--marginals": (["--marginals", j("M")], [j("M.sites.csv"), j("M.taxa.csv")]),
    }


def _read(path):
    with open(path, "rb") as f:
        return f.read()


@pytest.mark.gpu
@pytest.mark.parametrize("replay_selected", [False, True])
@pytest.mark.parametrize("manycd", [0, 1])
def test_cli_every_select_output_at_once_equals_each_alone(S, tmp_path, replay_selected, manycd):
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    write_txt(str(tmp_path / "g10s10.txt"), X, hard)
    base = [os.path.join(S.PKG_DIR, "mcmc"), "--chains", "64", "--burn", "20", "--samples", "60", "--seed", "0", "--select", "2",
            "--dataset", str(tmp_path / "g10s10.txt"), "--window", "16", "--manycd", str(manycd)]
    base += ["--replay-selected"] if replay_selected else []
    env = {k: v for k, v in os.environ.items() if k != "GSL_RNG_SEED"}

    def run(extra):
        out = subprocess.run(base + extra, check=True, capture_output=True, text=True, env=env, cwd=tmp_path).stdout.splitlines()
        assert out[0].startswith("chains 64 "), out  # the throughput line, whose timing differs from run to run
        return out[1:]

    (tmp_path / "all").mkdir()
    (tmp_path / "one").mkdir()
    together, alone = _outputs(tmp_path / "all"), _outputs(tmp_path / "one")
    out = run([a for args, _ in together.values() for a in args])
    want = out[:2]
    for flag, (args, files) in alone.items():
        lines = run(args)
        assert lines[:2] == out[:2], flag  # selection: and E[c]
        assert len(lines) == (2 if flag == "--po" else 3), (flag, lines)
        want += lines[2:]
        for mine, theirs in zip(together[flag][1], files):
            assert _read(mine) == _read(theirs), (flag, mine)
    assert out == want
    assert [next(h for h in HEADS if x.startswith(h)) for x in out] == list(HEADS)
