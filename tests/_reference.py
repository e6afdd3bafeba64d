"""What the unmodified reference program (oracle/_ref/agrep) answered, stored in tests/golden/reference_runs.json, so that the
tests that compare with it run on any checkout: the reference's sources are not part of this repository.

An answer is what a test reads from one run -- a count, the -n ordinals, a digest of stdout -- filed under the name of that
reading, the arguments and a sha-256 prefix of every input file.  An input that is not in the file is an error, never a skip.

To rewrite the file from the program itself (oracle/Makefile builds oracle/_ref where the reference sources are):
    AGB_RECORD_REFERENCE=1 python -m pytest tests/test_oracle_vs_reference.py tests/test_gpu_dropin.py -m "gpu or not gpu"
Only the answers asked for in that session are kept."""
import atexit, hashlib, json, os, subprocess, tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
BIN = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "agrep")
STORE = os.path.join(HERE, "golden", "reference_runs.json")
RECORD = os.environ.get("AGB_RECORD_REFERENCE") == "1"

_stored = None
_recorded = {}


def _key(what, args, files):
    args = [os.fsencode(a).decode("latin-1") for a in args]            # the bytes the program receives
    return json.dumps([what, args, [[name, hashlib.sha256(data).hexdigest()[:16]] for name, data in files]], separators=(",", ":"))


def _pack(v):
    """a list of ascending integers (ordinals) as runs: [1, 2, 3, 7] -> {"ints": "1-3,7"}"""
    if not (isinstance(v, list) and v and all(type(x) is int for x in v) and v == sorted(set(v))):
        return v
    runs = []
    for x in v:
        if runs and runs[-1][1] + 1 == x:
            runs[-1][1] = x
        else:
            runs.append([x, x])
    return {"ints": ",".join(str(a) if a == b else "%d-%d" % (a, b) for a, b in runs)}


def _unpack(v):
    if not (isinstance(v, dict) and "ints" in v):
        return v
    out = []
    for run in v["ints"].split(","):
        a, _, b = run.partition("-")
        out.extend(range(int(a), int(b or a) + 1))
    return out


def run(args, files):
    """(returncode, stdout, stderr) of the reference with ARGS followed by the names of FILES ([(name, bytes)]), run in a
    directory that holds just those files"""
    with tempfile.TemporaryDirectory(prefix="agb_ref_") as d:
        for name, data in files:
            with open(os.path.join(d, name), "wb") as f:
                f.write(data)
        p = subprocess.run([BIN] + list(args) + [name for name, _ in files], cwd=d, capture_output=True, timeout=120,
                           stdin=subprocess.DEVNULL)
    return p.returncode, p.stdout, p.stderr


def answer(what, args, files, read):
    """the stored value of read(returncode, stdout, stderr) for this run; with AGB_RECORD_REFERENCE=1, the program is run"""
    global _stored
    key = _key(what, args, files)
    if RECORD:
        if not os.path.exists(BIN):
            raise RuntimeError("AGB_RECORD_REFERENCE=1 needs %s (oracle/Makefile builds it from the reference sources)" % BIN)
        if not _recorded:
            atexit.register(_save)
        value = read(*run(args, files))
        _recorded[key] = _pack(value)
        return value
    if _stored is None:
        with open(STORE) as f:
            _stored = {json.dumps(row[:3], separators=(",", ":")): row[3] for row in json.load(f)}
    if key not in _stored:
        raise LookupError("no stored answer of the reference for %s; rewrite %s (see tests/_reference.py)" % (key, STORE))
    return _unpack(_stored[key])


def _save():
    with open(STORE, "w") as f:           # one answer per line: [what, args, [[file name, sha-256 prefix], ...], value]
        f.write("[\n" + ",\n".join(k[:-1] + "," + json.dumps(_recorded[k], separators=(",", ":")) + "]" for k in sorted(_recorded)) + "\n]\n")
