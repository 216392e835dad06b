"""Which options each `polypolish` subcommand accepts, and the usage errors of its argument parser (main.rs:23-126, plus the
additive --device, --gpus, --quiet and --host-parse and the `filter-polish` command).  An option a command does not take ends the
process with clap's exit code 2 and "unexpected argument"; one it takes gets past the parser, and with input files that do not
exist the command then fails at run time with exit code 1 (no usable GPU, or the missing file).  Needs no GPU."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "build", "polypolish")


@pytest.fixture(scope="module", autouse=True)
def built():
    import __graft_entry__ as g
    g.build()


# every option of the three commands, with a valid value where it takes one ({d}: a directory where nothing exists)
OPTIONS = {
    "--debug": ["{d}/debug.tsv"], "-i": ["0.2"], "--fraction_invalid": ["0.2"], "-v": ["0.5"], "--fraction_valid": ["0.5"],
    "-m": ["10"], "--max_errors": ["10"], "-d": ["5"], "--min_depth": ["5"], "--careful": [], "--gpus": ["1"],
    "--in1": ["{d}/in1.sam"], "--in2": ["{d}/in2.sam"], "--out1": ["{d}/out1.sam"], "--out2": ["{d}/out2.sam"],
    "--orientation": ["fr"], "--low": ["0.1"], "--high": ["99.9"],
    "--device": ["0"], "--quiet": [], "--host-parse": [],
}
POLISH = {"--debug", "-i", "--fraction_invalid", "-v", "--fraction_valid", "-m", "--max_errors", "-d", "--min_depth", "--careful", "--gpus"}
FILTER = {"--in1", "--in2", "--out1", "--out2", "--orientation", "--low", "--high"}
COMMON = {"--device", "--quiet", "--host-parse"}
ACCEPTS = {
    "polish": POLISH | COMMON,
    "filter": FILTER | COMMON,
    "filter-polish": (POLISH - {"--debug", "--gpus"}) | FILTER | COMMON,
}
# every required argument, naming files that do not exist
REQUIRED = {
    "polish": ["{d}/draft.fasta", "{d}/reads.sam"],
    "filter": ["--in1", "{d}/in1.sam", "--in2", "{d}/in2.sam", "--out1", "{d}/out1.sam", "--out2", "{d}/out2.sam"],
    "filter-polish": ["--in1", "{d}/in1.sam", "--in2", "{d}/in2.sam", "{d}/draft.fasta"],
}


def run(tmp_path, *args):
    d = str(tmp_path / "absent")
    r = subprocess.run([EXE] + [a.format(d=d) for a in args], capture_output=True, text=True, timeout=120)
    return r.returncode, r.stdout, r.stderr


@pytest.mark.parametrize("cmd", sorted(ACCEPTS))
@pytest.mark.parametrize("flag", sorted(OPTIONS))
def test_option_accepted_or_rejected(tmp_path, cmd, flag):
    required = REQUIRED[cmd]
    args = required if flag in required else [flag] + OPTIONS[flag] + required
    rc, out, err = run(tmp_path, cmd, *args)
    if flag in ACCEPTS[cmd]:
        assert rc == 1 and "unexpected argument" not in err and "Error: " in err, (rc, err)
    else:
        assert rc == 2 and "unexpected argument '%s' found" % flag in err, (rc, err)
    assert out == ""


@pytest.mark.parametrize("cmd", sorted(ACCEPTS))
def test_help_and_version(tmp_path, cmd):
    rc, out, err = run(tmp_path, cmd, "--help")
    assert rc == 0 and "Usage: polypolish %s" % cmd in out
    assert run(tmp_path, cmd, "-h")[:2] == (rc, out)
    rc, out, err = run(tmp_path, cmd, "-V", *REQUIRED[cmd])
    if cmd == "filter-polish":
        assert rc == 2 and "unexpected argument '-V' found" in err
    else:
        assert rc == 0 and out == "Polypolish-%s v0.6.1\n" % cmd


@pytest.mark.parametrize("cmd", sorted(ACCEPTS))
def test_value_forms(tmp_path, cmd):
    """`--name=value`, `-m5` / `-m=5` and everything after `--` being positional, as clap parses them."""
    if cmd != "filter":
        for form in (["--min_depth=5"], ["-d5"], ["-d=5"], ["-i", "0.2", "--max_errors=3"]):
            assert run(tmp_path, cmd, *form, *REQUIRED[cmd])[0] == 1, form
        rc, _, err = run(tmp_path, cmd, *REQUIRED[cmd], "--", "--careful")     # a SAM file named --careful, or a second <ASSEMBLY>
        assert rc == (1 if cmd == "polish" else 2), err
    else:
        assert run(tmp_path, cmd, "--low=0.5", "--orientation=rf", *REQUIRED[cmd])[0] == 1
        rc, _, err = run(tmp_path, cmd, *REQUIRED[cmd], "--", "--careful")
        assert rc == 2 and "unexpected argument '--careful' found" in err


@pytest.mark.parametrize("cmd,args,missing", [
    ("polish", [], "<ASSEMBLY>"),
    ("polish", ["--careful", "--quiet"], "<ASSEMBLY>"),
    ("filter", ["--in1", "a", "--in2", "b", "--out1", "c"], "--out2 <OUT2>"),
    ("filter", [], "--in1 <IN1>"),
    ("filter-polish", ["--in1", "a", "--in2", "b"], "<ASSEMBLY>"),
    ("filter-polish", ["--in1", "a", "x.fasta"], "--in2 <IN2>"),
    ("filter-polish", ["--in1", "a", "--in2", "b", "x.fasta", "y.fasta"], "<ASSEMBLY>"),
])
def test_missing_arguments(tmp_path, cmd, args, missing):
    rc, out, err = run(tmp_path, cmd, *args)
    assert rc == 2 and "the following required arguments were not provided" in err and missing in err, (rc, err)


@pytest.mark.parametrize("cmd", sorted(ACCEPTS))
def test_missing_and_invalid_values(tmp_path, cmd):
    for flag in sorted(ACCEPTS[cmd]):
        if not OPTIONS[flag]:
            continue
        rc, _, err = run(tmp_path, cmd, *REQUIRED[cmd], flag)
        assert rc == 2 and "a value is required for '" in err and "but none was supplied" in err, (flag, rc, err)
    for flag, bad in (("--min_depth", "x"), ("--max_errors", "-1"), ("--fraction_valid", "half"), ("--low", "one"), ("--device", "gpu")):
        if flag in ACCEPTS[cmd]:
            rc, _, err = run(tmp_path, cmd, flag, bad, *REQUIRED[cmd])
            assert rc == 2 and "invalid value '%s' for '%s" % (bad, flag) in err, (flag, rc, err)


def test_unknown_subcommand(tmp_path):
    rc, _, err = run(tmp_path, "polish-filter")
    assert rc == 2 and "unrecognized subcommand 'polish-filter'" in err
