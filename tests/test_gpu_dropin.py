"""The drop-in proof: the reference program linked against libagrepb200_dropin.so (oracle/_ref/agrep_dropin:
the reference's own main(), option parser, exec() and output(); only bitap/asearch/asearch0/asearch1/sgrep/
fill_buf come from this repo and run on the GPU) must print byte-for-byte what the unmodified reference
(oracle/_ref/agrep) prints.  oracle/Makefile builds both where the reference sources are; without them the drop-in cases
skip.  The stand-alone command line (agrep-b200) is checked against the reference's stdout stored in
tests/golden/reference_runs.json (tests/_reference.py), so it runs on any checkout."""
import hashlib, os, subprocess, tempfile
import pytest
import _corpus, _reference

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "agrep")
DROP = os.path.join(ROOT, "oracle", "_ref", "agrep_dropin")

from _corpus import overlap_text


def texts():
    return (("a.txt", _corpus.make_text(3000, seed=11)), ("b.txt", _corpus.make_text(2000, seed=12, trailing_newline=False)),
            ("para.txt", _corpus.make_text(2500, seed=13, paragraphs=True)),
            ("small.txt", _corpus.make_text(600, seed=14)),       # < 48 KiB: no block artefacts in -b (SURVEY 8c(1))
            ("semi.txt", _corpus.make_text(300, seed=15).replace(b"\n", b";").replace(b"the", b"Hello", 30).replace(b"and", b"xhello", 10) + b"last hello there"),   # (not "hello" at the very end: bm()'s sentinel copy of the pattern behind the text makes -w see a letter there)
            ("blank.txt", b"\n" * 3000 + b"one the two\n" + b"\n" * 3000 + b"x\n\n\ny"),   # more than half of the bytes close a record
            ("aba.txt", overlap_text("aba", 5)))      # a delimiter that overlaps itself, with chains ("abababa")


@pytest.fixture(scope="module")
def files():
    d = tempfile.mkdtemp(prefix="agb_dropin_")
    paths = {}
    for name, data in texts():
        paths[name] = os.path.join(d, name)
        open(paths[name], "wb").write(data)
    yield paths
    for p in paths.values():
        os.unlink(p)
    os.rmdir(d)


def run(binary, args, cwd=None):
    p = subprocess.run([binary] + args, capture_output=True, timeout=120, stdin=subprocess.DEVNULL, cwd=cwd)
    return p.returncode, p.stdout, p.stderr


def needs_dropin(*binaries):
    if not all(os.path.exists(b) for b in binaries):
        pytest.skip("the drop-in binaries link the reference's own objects: oracle/_ref is built only where its sources are")


CASES = [
    (["-c", "the"], ["a.txt"]),                                  # sgrep -> bm, count
    (["the"], ["a.txt"]),                                        # sgrep -> bm, records printed
    (["-c", "the"], ["a.txt", "b.txt"]),                         # two files: "file: N" lines
    (["-h", "government"], ["a.txt", "b.txt"]),
    (["-l", "government"], ["a.txt", "b.txt"]),
    (["-w", "-c", "the"], ["b.txt"]),
    (["-n", "because each"], ["a.txt"]),                         # bitap exact, line numbers
    (["-n", "-1", "because each"], ["a.txt"]),                   # asearch
    (["-n", "-2", "-i", "Government"], ["a.txt", "b.txt"]),
    (["-c", "-n", "-3", "government"], ["a.txt"]),
    (["-n", "-5", "governmental"], ["a.txt"]),                   # asearch0
    (["-n", "-2", "-S2", "between both"], ["a.txt"]),            # asearch1
    (["-n", "-v", "-1", "the"], ["b.txt"]),                      # inverse
    (["-c", "-n", "-v", "the"], ["a.txt"]),
    (["-n", "-w", "-1", "matching"], ["a.txt"]),
    (["-n", "st.t[a-e]"], ["a.txt"]),
    (["-n", "-b", "-1", "homogeneous"], ["small.txt"]),
    (["-n", "-d", "$$", "-1", "because each"], ["para.txt"]),    # paragraph records
    (["-c", "-n", "-d", "$$", "-w", "world"], ["para.txt"]),
    (["-n", "-y", "-B", "goverment of the peple"], ["a.txt"]),   # best-match sweep, no prompt
    (["-n", "-L2", "-1", "the"], ["a.txt"]),                     # output limit
    (["-s", "the"], ["a.txt"]),
    (["-n", "^the"], ["a.txt"]),
    (["-n", "world$"], ["b.txt"]),
    (["-n", "a#d;world"], ["a.txt"]),
    (["-d", ";", "hello"], ["semi.txt"]),                        # sgrep keeps its engine under -d: ASCII case folded, bm() record cut
    (["-c", "-d", ";", "hello"], ["semi.txt"]),
    (["-c", "-w", "-d", ";", "hello"], ["semi.txt"]),
    (["-n", "-v", "zzz"], ["blank.txt"]),                        # every blank line is a reported record (list longer than n/2)
    (["-c", "-n", "^$"], ["blank.txt"]),
    (["-n", "-d", "aba", "-1", "state"], ["aba.txt"]),           # occurrences taken from the left, overlapping ones dropped
    (["-c", "-n", "-d", "aba", "e"], ["aba.txt"]),
    (["-n", "-1", "^$"], ["blank.txt"]),
]


@pytest.mark.parametrize("args,names", CASES)
def test_same_stdout_as_reference(files, args, names):
    needs_dropin(REF, DROP)
    fl = [files[n] for n in names]
    r = run(REF, ["-V0"] + args + fl)
    d = run(DROP, ["-V0"] + args + fl)
    assert d[2].replace(b"agrep_dropin", b"agrep") == r[2], (d[2], r[2])
    assert d[1] == r[1]
    assert d[0] == r[0]


CLI = os.path.join(ROOT, "agrep_b200", "agrep-b200")
CLI_CASES = [c for c in CASES if not any(a in ("-L2", "-s") or a.startswith("-S") for a in c[0]) and c[0][-1] not in ("a#d;world",)
             and "semi.txt" not in c[1]]


@pytest.mark.parametrize("args,names", CLI_CASES)
def test_standalone_cli_prints_what_the_reference_prints(files, args, names):
    """agrep-b200 (agrep_b200/csrc/agrep_main.c): our own main() + output() restatement over the engine.  Both run where
    the files are, on their bare names (names are part of the output): exit code, length and sha-256 of stdout."""
    data = dict(texts())
    summary = lambda rc, out, err: [rc, len(out), hashlib.sha256(out).hexdigest()]
    r = _reference.answer("rc_stdout_size_sha256", args, [(n, data[n]) for n in names], summary)   # default verbosity: with the "Grand Total" line
    d = summary(*run(CLI, args + names, cwd=os.path.dirname(files[names[0]])))
    assert d[1:] == r[1:]
    assert d[0] == r[0]


MEM = os.path.join(ROOT, "oracle", "_ref", "memagrep_cli")
MEMDROP = os.path.join(ROOT, "oracle", "_ref", "memagrep_dropin_cli")


@pytest.mark.parametrize("args,name", [(["-n", "-1", "because each"], "a.txt"), (["-c", "-n", "-1", "the"], "a.txt"),
                                       (["-c", "-n", "-1", "the"], "b.txt"), (["-n", "-2", "governmental"], "b.txt"),
                                       (["-c", "-n", "the"], "b.txt"), (["-n", "-w", "-d", "$$", "world"], "para.txt")])
def test_memory_mode_through_the_dropin(files, args, name):
    """memagrep() (agrep.c:3282; scan loop bitap.c:309-446): the reference's in-memory entry point with the scan objects
    replaced by the drop-in layer (fd == -1: the caller's buffer is scanned, no delimiter is appended behind it, so an
    undelimited last record is not reported -- by -c either) prints and returns what the unmodified one does."""
    needs_dropin(MEM, MEMDROP)
    r = run(MEM, [files[name], "-V0"] + args)
    d = run(MEMDROP, [files[name], "-V0"] + args)
    assert d[1] == r[1] and d[0] == r[0]


def test_three_gib_file_streams_through_the_dropin(tmp_path):
    """`agrep_dropin -c` on a file of 3 GiB (past the reference's 2 GiB `int` offsets): the file is pread(2) straight into
    the pinned ring and on to the device, never slurped -- same count as the unmodified reference, resident set what the
    same binary takes on a 1 MiB file (CUDA context and module: 2.0 - 2.7 GB from box to box) plus less than a third of
    the file.  Skipped where the scratch disk or the page cache cannot hold the file."""
    import resource, shutil, sys
    sys.path.insert(0, ROOT)
    import agrep_b200 as ag
    needs_dropin(REF, DROP)
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > (5 << 30) else str(tmp_path)
    if shutil.disk_usage(base).free < (4 << 30):
        pytest.skip("no room for a 3 GiB file")
    path = os.path.join(base, "agb_big_%d.txt" % os.getpid())
    piece, total = 256 << 20, 3 << 30
    try:
        with open(path, "wb") as f:
            for i in range(total // piece):
                f.write(ag.corpus_host(piece, first_page=i * (piece // 4096), needle="because each", needle_every=512, needle_maxedits=3))
        small = path + ".small"
        with open(small, "wb") as f:
            f.write(ag.corpus_host(1 << 20, needle="because each", needle_every=512, needle_maxedits=3))
        proc = subprocess.Popen([DROP, "-V0", "-c", "-2", "because each", small], stdout=subprocess.PIPE, stderr=subprocess.PIPE, stdin=subprocess.DEVNULL)
        proc.stdout.read(); proc.stderr.read()
        _, _, ru = os.wait4(proc.pid, 0)
        small_rss_kib = ru.ru_maxrss
        os.unlink(small)
        for args in (["-c", "-n", "-2", "because each"], ["-c", "government"]):
            r = subprocess.run([REF, "-V0"] + args + [path], capture_output=True, timeout=900)
            # this child's own peak resident set (wait4), not the running maximum over every child of the test process
            proc = subprocess.Popen([DROP, "-V0"] + args + [path], stdout=subprocess.PIPE, stderr=subprocess.PIPE, stdin=subprocess.DEVNULL)
            out, errtxt = proc.stdout.read(), proc.stderr.read()          # (-c: a few bytes each)
            _, _, ru = os.wait4(proc.pid, 0)
            rss_kib = ru.ru_maxrss
            assert out == r.stdout and int(out.split()[0]) > 1000, (args, out, r.stdout, errtxt[-300:])
            # CUDA context + module + pinned ring + libraries (2.0 - 2.7 GB from box to box), not the file: the same binary on
            # a 1 MiB file takes as much
            assert rss_kib * 1024 < small_rss_kib * 1024 + total // 3, (rss_kib, small_rss_kib)
        # records past 2 GiB come out with the right bytes: the last matching lines of the file, as the reference prints them
        r = subprocess.run("%s -V0 -2 'because each' %s | tail -c 4096" % (REF, path), shell=True, capture_output=True, timeout=900)
        d = subprocess.run("%s -V0 -2 'because each' %s | tail -c 4096" % (DROP, path), shell=True, capture_output=True, timeout=900)
        assert d.stdout == r.stdout and len(d.stdout) > 100
    finally:
        try:
            os.unlink(path)
        except OSError:
            pass
