#!/usr/bin/env python
"""
Golden fixtures for the drop-in surface (CLI, features .csv loader, *_reads.csv / compiled.csv /
compiled_stats.csv): runs the UNMODIFIED reference CLI (`python -m fast2q -c ...` from the checkout refharness.py
points at, with the colorama / matplotlib stubs of tests/golden/_stubs) on the input folders of tests/cli_golden.py
and stores its outputs in tests/golden/cli_cases.json.gz with what tests/cli_golden.py needs to regenerate and check
the inputs (cli_golden.file_entry).  Needs the reference checkout:

    python tests/golden/make_cli_golden.py

Also stores the reference's features_loader() result for a few awkward library files and the reference's
input_parser() dict for a few command lines.
"""
import glob
import gzip
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import cli_golden  # noqa: E402
import refharness  # noqa: E402


def run_reference_cli(case):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(HERE, "_stubs"), refharness.REF_ROOT]), PYTHONWARNINGS="ignore")
    with tempfile.TemporaryDirectory() as td:
        src, outd = os.path.join(td, "in"), os.path.join(td, "out")
        os.makedirs(src); os.makedirs(outd)
        for fn, data in case["files"].items():
            open(os.path.join(src, fn), "wb").write(data)
        args = ["-c", "--s", src, "--o", outd] + case["args"]
        if case["library"] is not None:
            lp = os.path.join(td, "library.csv")
            open(lp, "w").write(case["library"])
            args += ["--g", lp]
        p = subprocess.run([sys.executable, "-m", "fast2q"] + args, env=env, cwd=td, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-2000:]
        dirs = glob.glob(os.path.join(outd, "2FAST2Q_output_*"))
        assert len(dirs) == 1
        outs = {}
        for f in sorted(os.listdir(dirs[0])):
            if f.endswith(".csv"):
                outs[f] = open(os.path.join(dirs[0], f), newline="").read().replace(td, "<TMP>")
        return outs, p.stdout.replace(td, "<TMP>")


def loader_cases():
    """library files that exercise features_loader's quirks (fast2q.py:125-186)"""
    return {
        "comma": "a,ACGT\nb,acgt t\nc,GGGG\nb,TTTT\n",
        "semicolon": "x;AAAA\ny;CCCC\n",
        "tab": "x\tAAAA\ny\tCCCC\n",
        "comma_then_short_line": "a,ACGT\nb,CCCC\nbroken\nc,GGGG\n",
        "mixed_separators": "a,ACGT\nb;CCCC\nc\tGGGG\n",
        "three_columns": "a,ACGT,extra\nb,CCCC,more\n",
        "semicolon_with_commas_in_name": "n,1;ACGT\nm,2;CCCC\n",
        "crlf": "a,ACGT\r\nb,CCCC\r\n",
        "blank_last_line": "a,ACGT\nb,CCCC\n\n",
        "header_like": "name,sequence\ng1,ACGTAC\n",
        "trailing_space_after_seq": "a,ACGT \nb, CCCC\n",
    }


def parser_cases():
    return [
        ["-c"],
        ["-c", "--s", "/data/in", "--g", "/data/lib.csv", "--o", "/data/out"],
        ["-c", "--s", "/d", "--g", "/l.csv", "--o", "/o", "--m", "2", "--ph", "25", "--st", "3,40", "--l", "18", "--pb", "--k", "--fs",
         "--cp", "3", "--fn", "xyz"],
        ["-c", "--s", "/d", "--o", "/o", "--mo", "ec", "--us", "acgt", "--ds", "TTGA", "--msu", "1", "--msd", "2", "--qsu", "10",
         "--qsd", "0"],
        ["-c", "--s", "/d", "--g", "/l.csv", "--o", "/o", "--mo", "Counter", "--fn"],
    ]


def main():
    assert refharness.available()
    ref = refharness.load()
    out = dict(cli=[], loader={}, parser=[])
    for c in cli_golden.cli_inputs():
        outs, stdout = run_reference_cli(c)
        out["cli"].append(dict(name=c["name"], args=c["args"], library=c["library"],
                               files={k: cli_golden.file_entry(k, v) for k, v in c["files"].items()}, outputs=outs))
        print(c["name"], {k: len(v) for k, v in outs.items()})
    for name, text in loader_cases().items():
        with tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False) as f:
            f.write(text)
        try:
            feats = ref.features_loader(f.name)
            res = [[seq, v.name] for seq, v in feats.items()]
        except SystemExit:
            res = "FATAL"
        os.unlink(f.name)
        out["loader"][name] = dict(text=text, expect=res)
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as td:
        os.chdir(td)                                     # an empty cwd: no stray .csv for the --g default
        for argv in parser_cases():
            old = sys.argv
            sys.argv = ["2fast2q"] + argv
            try:
                p = ref.input_parser()
            finally:
                sys.argv = old
            out["parser"].append(dict(argv=argv, expect={k: (v.replace(td, "<CWD>") if isinstance(v, str) else v) for k, v in p.items()}))
        os.chdir(cwd)
    with gzip.GzipFile(os.path.join(HERE, "cli_cases.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(out).encode())
    print("written", os.path.getsize(os.path.join(HERE, "cli_cases.json.gz")))


if __name__ == "__main__":
    main()
