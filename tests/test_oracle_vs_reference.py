"""Pins oracle/agrep_oracle.c against the UNMODIFIED reference (oracle/_ref/agrep, built by oracle/Makefile), through
its answers stored in tests/golden/reference_runs.json (tests/_reference.py).  Reference invocations follow SURVEY.md 8(c):
k>0 automaton forced with -n, unit-cost asearch1 with -S1, simple literals via sgrep/bm."""
import random, re
import pytest
import _oracle, _corpus, _reference


def ref(what, args, data, read):
    return _reference.answer(what, ["-V0"] + args, [("text.txt", data)], read)


def ref_count(args, data):
    return ref("count", ["-c"] + args, data, lambda rc, out, err: int(out.strip()) if out.strip() else 0)


def ordinals(out, pattern=rb"^(\d+): "):
    return [int(m.group(1)) for m in re.finditer(pattern, out, re.M)]


def ref_ordinals(args, data):
    return ref("ordinals", ["-n"] + args, data, lambda rc, out, err: ordinals(out))


TEXT = _corpus.make_text(4000, seed=12345)
TEXT_NONL = _corpus.make_text(500, seed=7, trailing_newline=False)
PARA = _corpus.make_text(3000, seed=99, paragraphs=True)

CASES = [
    # (pattern, oracle kwargs, reference args)
    ("because each", dict(k=0, linenum=1), []),
    ("because each", dict(k=1, linenum=1), ["-1"]),
    ("because each", dict(k=2, linenum=1), ["-2"]),
    ("government", dict(k=3, linenum=1), ["-3"]),
    ("governmental", dict(k=4, linenum=1, nocase=1), ["-4", "-i"]),
    ("governmental", dict(k=5, linenum=1), ["-5"]),
    ("homogeneous approx", dict(k=8, linenum=1), ["-8"]),
    ("matching", dict(k=1, linenum=1, wordbound=1), ["-1", "-w"]),
    ("the", dict(k=0, linenum=1, wordbound=1), ["-w"]),
    ("pattern string", dict(k=2, linenum=1, inverse=1), ["-2", "-v"]),
    ("pat[a-t]ern", dict(k=1, linenum=1), ["-1"]),
    ("st.ing", dict(k=0, linenum=1), []),
    ("<algo>rithm", dict(k=2, linenum=1), ["-2"]),
    ("^the", dict(k=0, linenum=1), []),
    ("world$", dict(k=1, linenum=1), ["-1"]),
    ("state;world", dict(k=0, linenum=1), []),
    ("[^a-s]he ", dict(k=0, linenum=1), []),
    ("between both life", dict(k=2, linenum=1, cost_s=1), ["-2", "-S1"]),
    ("between both life", dict(k=3, linenum=1, cost_s=2), ["-3", "-S2"]),
    ("between both life", dict(k=3, linenum=1, cost_i=2, cost_d=3), ["-3", "-I2", "-D3"]),
    ("government", dict(k=2, linenum=1, ins_free=1), ["-2", "-p"]),
    ("a#t", dict(k=0, linenum=1), []),
]


@pytest.mark.parametrize("pattern,okw,rargs", CASES)
@pytest.mark.parametrize("which", ["nl", "nonl"])
def test_automaton_matches_reference(pattern, okw, rargs, which):
    data = TEXT if which == "nl" else TEXT_NONL
    a = _oracle.compile(pattern, width=32, **okw)
    cnt, recs = _oracle.scan(a, data)
    assert cnt == ref_count(["-n"] + rargs + [pattern], data)
    # -n prints j-1 (agrep.c:3878)
    assert [r[2] - 1 for r in recs] == ref_ordinals(rargs + [pattern], data)


@pytest.mark.parametrize("pattern,k", [("win", 0), ("because each", 2), ("state", 1)])
def test_paragraph_records(pattern, k):
    a = _oracle.compile(pattern, width=32, k=k, linenum=1, wordbound=1, delim="$$")
    cnt, recs = _oracle.scan(a, PARA)
    assert cnt == ref_count(["-n", "-w", "-d", "$$", "-%d" % k, pattern] if k else ["-n", "-w", "-d", "$$", pattern], PARA)


@pytest.mark.parametrize("pattern,kw,rargs", [
    ("the", {}, []), ("The", {}, []), ("government", {}, []), ("the", dict(wordbound=1), ["-w"]),
    ("each", dict(nocase=1), ["-i"]), ("zzzz", {}, [])])
@pytest.mark.parametrize("which", ["nl", "nonl"])
def test_sgrep_bm_counts(pattern, kw, rargs, which):
    """config 1: `agrep -c the` goes through sgrep()->bm() (case-insensitive substring, once per line)."""
    data = TEXT if which == "nl" else TEXT_NONL
    a = _oracle.compile(pattern, **kw)
    assert a.engine == 4
    cnt, _ = _oracle.scan(a, data, want_records=False)
    assert cnt == ref_count(rargs + [pattern], data)


@pytest.mark.parametrize("pattern,delim,kw,rargs", [
    ("hello", ";", {}, []), ("HELLO", ";", {}, []), ("hello", ";", dict(wordbound=1), ["-w"]), ("each", "@#", {}, []),
    ("state", ";", dict(nocase=1), ["-i"]), ("because each", "%", {}, []),
    ("homogeneous approximate matching", ";", {}, []),          # > 20 characters: monkey() instead of bm() (sgrep.c:407-442, 1540)
])
def test_sgrep_keeps_its_engine_under_d(pattern, delim, kw, rargs):
    """checksg() does not look at -d: a simple literal at k=0 still goes to sgrep()/bm() -- ASCII case folded whatever -i
    says -- and bm() cuts the records with backward_/forward_delimiter() (sgrep.c:775-795)."""
    body = TEXT[:30000].replace(b"\n", delim.encode(), 400).replace(b"the", b"Hello", 40).replace(b"and", b"xhello", 20)
    for data in (b"Hello world;foo bar;HELLO again;nothing".replace(b";", delim.encode()), body, delim.encode() + body, body + delim.encode()):
        a = _oracle.compile(pattern, delim=delim, **kw)
        assert a.engine == 4
        cnt, _ = _oracle.scan(a, data, want_records=False)
        assert cnt == ref_count(rargs + ["-d", delim, pattern], data), (pattern, delim, data[:40])


@pytest.mark.parametrize("pattern", ["the of and to in that is was he for", "homogeneous approximate matching", "governmental homogeneous"])
def test_sgrep_long_literals_take_monkey(pattern):
    """m > 20 (LONG_EXAC): the reference runs monkey() instead of bm() (sgrep.c:407-442, 1540-1834); same record semantics"""
    data = TEXT + (b"xx " + pattern.encode() + b" yy\n") * 3 + pattern.upper().encode() + b"\n" + TEXT[:5000]
    a = _oracle.compile(pattern)
    assert a.engine == 4 and a.litlen > 20
    cnt, _ = _oracle.scan(a, data, want_records=False)
    assert cnt >= 4 and cnt == ref_count([pattern], data)


def test_latin1_fold_is_the_table_the_reference_ends_up_with():
    """-i at k=0 reads bytes through LUT[] (bitap.c:171) = CP[ISO-8859-1].lower_1 with the metasymbol bytes put back to
    themselves (agrep.c:2835-2848): 0xC9 folds to 0xE9, but 0x83 does not fold to 'f', 0x8f not to 0x86, 0x99 not to 0x94"""
    data = b"\x83ood one\nfood two\nab\x99cd\nab\x94cd\ncaf\xc9 x\ncaf\xe9 y\nq\x8fq\nq\x86q\n"
    for pat in (b"food", b"b\x94c", b"caf\xe9", b"q\x86q", b"\x83ood", b"b\x99c"):
        a = _oracle.compile(pat, k=0, linenum=1, nocase=1)
        cnt, recs = _oracle.scan(a, data)
        assert [r[2] - 1 for r in recs] == ref_ordinals(["-i", pat], data), pat


def test_random_differential():
    """SURVEY appendix A differential driver: random substrings with 0-2 edits, k in 1..3, -n forced."""
    rnd = random.Random(2024)
    lines = TEXT.decode().split("\n")
    for trial in range(40):
        ln = rnd.choice([l for l in lines if len(l) > 40])
        m = rnd.choice([4, 6, 8, 12, 16, 20, 24, 27])
        st = rnd.randrange(len(ln) - m)
        pat = _corpus.mutate(rnd, ln[st:st + m], rnd.randint(0, 2))
        if any(ch in pat for ch in ";,.*-[]()<>|#{}~^$\\"):
            continue
        k = rnd.randint(1, 3)
        if len(pat) <= k:
            continue
        a = _oracle.compile(pat, width=32, k=k, linenum=1)
        cnt, recs = _oracle.scan(a, TEXT)
        assert [r[2] - 1 for r in recs] == ref_ordinals(["-%d" % k, pat], TEXT), (pat, k)


def test_pattern_too_long_matches_reference_limit():
    # maskgen.c:201-208: literal of 30 chars -> M = 32 -> rejected at width 32; fine at width 64
    with pytest.raises(_oracle.OracleError):
        _oracle.compile("a" * 30, width=32, k=1, linenum=1)
    _oracle.compile("a" * 29, width=32, k=1, linenum=1)
    _oracle.compile("a" * 40, width=64, k=1, linenum=1)


def test_random_metachar_differential():
    """random patterns with classes, '.', '#', <>, ',' and ';', anchors, under -i/-w/-v/-p/-S2 and user delimiters, on a
    text shorter than one 48 KiB block (no block artefacts): ordinals of the matching lines (newline records), counts
    (user delimiters: their records are not one per output line).  Cases the reference refuses are skipped."""
    base = _corpus.make_text(400, seed=5)
    words = [w for w in base.decode().split() if w.isalpha()]
    rnd = random.Random(31)

    def rand_pattern():
        w = (rnd.choice(words) + " " + rnd.choice(words))[:rnd.randint(3, 14)]
        out = []
        for ch in w:
            r = rnd.random()
            out.append("." if r < 0.08 else "[" + ch + "x]" if r < 0.12 else "[^q]" if r < 0.15 else "#" if r < 0.17
                       else ch.upper() if r < 0.19 else ch)
        p = "".join(out)
        r = rnd.random()
        return ("<" + p[:2] + ">" + p[2:] if r < 0.08 else p + "," + rnd.choice(words) if r < 0.14
                else p + ";" + rnd.choice(words) if r < 0.20 else "^" + p if r < 0.24 else p + "$" if r < 0.28 else p)
    compared = 0
    for _ in range(160):
        data = ("\n".join(base.decode().split("\n")[:rnd.randint(200, 390)]) + rnd.choice(["\n", "", "\n\n"])).encode()
        pat = rand_pattern()
        k = rnd.choice([0, 0, 1, 2, 3, 4, 6])
        kw, args = dict(k=k, linenum=1), (["-%d" % k] if k else [])
        for p_, key, flag in ((0.25, "nocase", "-i"), (0.15, "wordbound", "-w"), (0.1, "inverse", "-v"), (0.05, "ins_free", "-p")):
            if rnd.random() < p_:
                kw[key] = 1; args.append(flag)
        if rnd.random() < 0.15:
            kw["delim"] = rnd.choice(["$$", "e "]); args += ["-d", kw["delim"]]
        if k and rnd.random() < 0.06:
            kw["cost_s"] = 2; args.append("-S2")
        try:
            a = _oracle.compile(pat, width=32, **kw)
        except _oracle.OracleError:
            continue
        cnt, recs = _oracle.scan(a, data)
        if "delim" in kw:
            out = ref("count_if_accepted", ["-c", "-n"] + args + [pat], data,
                      lambda rc, out, err: int(out.strip()) if out.strip().isdigit() else None)
            if out is not None:
                assert out == cnt, (pat, args)
                compared += 1
            continue
        out = ref("ordinals_if_accepted", ["-n"] + args + [pat], data,
                  lambda rc, out, err: None if rc == 255 or err.strip() else ordinals(out))
        if out is None:
            continue
        assert [r[2] - 1 for r in recs] == out, (pat, args)
        compared += 1
    assert compared > 100


from _corpus import overlap_text


@pytest.mark.parametrize("delim", ["aba", "abab", "=-=", "e e", "xyx"])
@pytest.mark.parametrize("pattern,kw,rargs", [("state", dict(k=1, linenum=1), ["-1"]), ("e", dict(k=0, linenum=1), []),
                                              ("world", dict(k=0, linenum=1, inverse=1), ["-v"])])
def test_self_overlapping_delimiters(delim, pattern, kw, rargs):
    """a delimiter that overlaps itself: the automaton takes occurrences from the left and drops those that share a byte with
    one it took (asearch.c:55-57, 175-186) -- count and ordinals of the restatement against the reference binary"""
    for seed in (3, 4):
        data = overlap_text(delim, seed)
        for d in (data, delim.encode() + data, data + delim.encode(), data[:-len(delim)] + delim.encode()[:-1]):
            a = _oracle.compile(pattern, delim=delim, **kw)
            cnt, recs = _oracle.scan(a, d)
            assert cnt > 3
            assert cnt == ref_count(["-n"] + rargs + ["-d", delim, pattern], d), (delim, pattern)
            out = ref("record_numbers", ["-n"] + rargs + ["-d", delim, pattern], d, lambda rc, out, err: ordinals(out, rb"(\d+): "))
            # (with a user delimiter -n prints j itself: the record count starts one lower, bitap.c:151-156 / agrep.c:3878)
            assert [r[2] for r in recs] == out, (delim, pattern)


@pytest.mark.parametrize("pattern,kw,rargs", [("because each", dict(k=2, linenum=1), ["-2"]), ("state", dict(k=0, linenum=1), []),
                                              ("gov[ea]rnment", dict(k=1, linenum=1), ["-1"]), ("world", dict(k=1, linenum=1, wordbound=1), ["-1", "-w"])])
def test_inverse_count_is_records_minus_matches(pattern, kw, rargs):
    """what the device's complement count rests on (scan.cu complement_usable): under -v every newline record either matches
    or does not, so `-c -v` = records - `-c`, with records = newlines + one for an unterminated last line -- checked on the
    reference binary itself and on the restatement, for texts with blank lines, without a final newline, starting with
    newlines, ending in a match"""
    body = TEXT[:40000]
    for data in (body, body[:-1], b"\n\n" + body, body.replace(b"the\n", b"the\n\n\n", 40), body + b"because each", body + b"\n\n\n", b"\n", b"x"):
        records = data.count(b"\n") + (0 if data.endswith(b"\n") else 1)
        pos = ref_count(["-n"] + rargs + [pattern], data)
        inv = ref_count(["-n", "-v"] + rargs + [pattern], data)
        assert inv == records - pos, (pattern, len(data), inv, records, pos)
        a = _oracle.compile(pattern, inverse=1, **kw)
        assert _oracle.scan(a, data, want_records=False)[0] == inv
