"""loader of tests/golden/cli_cases.json.gz (made by tests/golden/make_cli_golden.py from the unmodified reference).

The input folders are regenerated here from the seeded generator (2fast2q_b200/synth.py); the golden file keeps the sha256
of each file's content (gunzipped for a .gz file) and the reference's outputs.  A gzip file that breaks off before its end
is stored verbatim: where it stops lies in its compressed bytes."""
import base64
import gzip
import hashlib
import importlib
import io
import json
import os
import re

_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cli_cases.json.gz")
_cache = None
_inputs = None


def gz(data: bytes, level=6) -> bytes:
    b = io.BytesIO()
    with gzip.GzipFile(fileobj=b, mode="wb", compresslevel=level, mtime=0) as f:
        f.write(data)
    return b.getvalue()


def cli_inputs():
    """the six input folders the reference CLI was run on: name, library text, files {name: bytes}, arguments"""
    synth = importlib.import_module("2fast2q_b200.synth")
    out = []
    # 1. Counter, fixed position, three files (.fastq, .fastq.gz, CRLF .fastq), numeric names, awkward library file
    names, keys = synth.make_library(2, 150, 20)
    spec = synth.default_spec(2)
    lib_lines = []
    for i, k in enumerate(keys):
        s = k.decode()
        if i == 7:
            s = s.lower()
        if i == 9:
            s = s[:10] + " " + s[10:]
        lib_lines.append(f"{i + 1},{s}")
    lib_lines.insert(20, f"999,{keys[3].decode()}")            # shares its sequence with entry 4: ignored with a warning
    # (a repeated NAME makes the reference itself crash in run_stats, fast2q.py:1475, so none is used here)
    reads = synth.fixed_reads(keys, 0, 5400, **spec).tobytes()
    rec = 118
    c = reads[5000 * rec:5400 * rec].replace(b"\n", b"\r\n")
    out.append(dict(name="cli_counter", library="\n".join(lib_lines) + "\n",
                    files={"sampleA.fastq": reads[:3000 * rec], "sampleB.fastq.gz": gz(reads[3000 * rec:5000 * rec]),
                           "sampleC.fastq": c},
                    args=["--m", "1", "--ph", "30", "--k", "--pb", "--cp", "2"]))
    # 2. Extract + Count between delimiters with mismatches, two files
    bs = synth.barseq_reads(4, 3000)
    cut = bs.find(b"\n@", len(bs) // 2) + 1
    out.append(dict(name="cli_ec", library=None, files={"bar1.fastq": bs[:cut], "bar2.fastq.gz": gz(bs[cut:])},
                    args=["--mo", "EC", "--us", "GTTCAGAGTTCT", "--ds", "CTGAATAGGCCA", "--msu", "1", "--msd", "1", "--pb", "--k",
                          "--cp", "2"]))
    # 3. dual fixed windows, ';' separated library, alphabetical names, custom file name, intermediates deleted
    dn, dk, xs, ys = synth.dual_library(5, 120)
    dr = synth.dual_reads(5, 2400, xs, ys, mode="fixed")
    cut = dr.find(b"\n@", len(dr) // 3) + 1
    out.append(dict(name="cli_dual", library="".join(f"{n};{k.decode()}\n" for n, k in zip(dn, dk)),
                    files={"d_one.fastq": dr[:cut], "d_two.fastq": dr[cut:]},
                    args=["--st", "0,30", "--l", "20", "--m", "1", "--pb", "--cp", "2", "--fn", "mycounts"]))
    # 4. a single file: File-Split mode is forced (fast2q.py:1671-1672); --cp 1 keeps the reference's chunking exact
    out.append(dict(name="cli_single_split", library="".join(f"{n},{k.decode()}\n" for n, k in zip(names, keys)),
                    files={"only.fastq.gz": gz(reads[:2000 * rec])}, args=["--m", "2", "--pb", "--k", "--cp", "1"]))
    # 5. a gzip file cut off mid-stream: warning + partial counts (fast2q.py:405-407)
    whole = gz(reads[:2500 * rec])
    out.append(dict(name="cli_truncated_gz", library="".join(f"{n},{k.decode()}\n" for n, k in zip(names, keys)),
                    files={"good.fastq": reads[2500 * rec:3500 * rec], "cut.fastq.gz": whole[: len(whole) * 6 // 10]},
                    args=["--pb", "--k", "--cp", "2"]))
    # 6. delimiter pairs in Counter mode, tab separated library
    n5, k5, xs5, ys5 = synth.dual_library(5, 100)
    d5 = synth.dual_reads(5, 1500, xs5, ys5, mode="delim")
    cut = d5.find(b"\n@", len(d5) // 2) + 1
    out.append(dict(name="cli_dual_delim", library="".join(f"{n}\t{k.decode()}\n" for n, k in zip(n5, k5)),
                    files={"p1.fastq": d5[:cut], "p2.fastq": d5[cut:]},
                    args=["--us", "ACCGGT,GGATCC", "--ds", "TTGACA,CAATTG", "--m", "1", "--pb", "--k", "--cp", "2"]))
    return out


def file_entry(fn, data):
    """what the golden file keeps of one input file"""
    try:
        content = gzip.decompress(data) if fn.endswith(".gz") else data
    except EOFError:
        return {"base64": base64.b64encode(data).decode()}
    return {"sha256": hashlib.sha256(content).hexdigest()}


def load():
    global _cache
    if _cache is None:
        with gzip.open(_PATH, "rb") as f:
            _cache = json.loads(f.read().decode())
    return _cache


def case(name):
    return [c for c in load()["cli"] if c["name"] == name][0]


def input_files(c):
    """{file name: bytes} of a golden case: regenerated, and checked against what the reference was given"""
    global _inputs
    if _inputs is None:
        _inputs = {x["name"]: x["files"] for x in cli_inputs()}
    files = {}
    for fn, entry in c["files"].items():
        if "base64" in entry:
            files[fn] = base64.b64decode(entry["base64"])
        else:
            files[fn] = _inputs[c["name"]][fn]
            assert file_entry(fn, files[fn]) == entry, f"{c['name']}/{fn}: the generator no longer makes the input the reference read"
    return files


def write_inputs(c, root):
    """creates <root>/in/* (+ <root>/library.csv); returns the reference-style argv"""
    src, out = os.path.join(root, "in"), os.path.join(root, "out")
    os.makedirs(src, exist_ok=True)
    os.makedirs(out, exist_ok=True)
    for fn, data in input_files(c).items():
        with open(os.path.join(src, fn), "wb") as f:
            f.write(data)
    argv = ["-c", "--s", src, "--o", out] + list(c["args"])
    if c["library"] is not None:
        with open(os.path.join(root, "library.csv"), "w", newline="") as f:
            f.write(c["library"])
        argv += ["--g", os.path.join(root, "library.csv")]
    return argv


_TIME = re.compile(r"ran in \S+ \S+ for file")


def mask_reads_csv(text):
    """the statistics sentence without its wall-clock part"""
    return _TIME.sub("ran in <T> for file", text)


def mask_stats_csv(text, tmp=None):
    """compiled_stats.csv without run times and without the '#cmd used' line (paths / added flags differ)"""
    out = []
    for line in text.split("\r\n"):
        if line.startswith("#cmd used") or line.startswith('"#cmd used'):
            continue
        cols = line.split(",")
        if not line.startswith("#") and not line.startswith('"#') and len(cols) == 9:
            cols[1], cols[2] = "<T>", "<U>"
            line = ",".join(cols)
        out.append(line)
    return "\r\n".join(out)
