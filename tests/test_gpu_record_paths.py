"""Record paths that only size, density or workspace history reach, against the oracle: the candidate list that
overflows and the record stage that runs again (a bigger list, or every byte), lists cut short by the caller's capacity
in every emit form, -B lists on one device, and the streamed host entry with its 64 MiB slice edges placed on an anchor,
on a closing newline and inside a '$$' run.

Large texts are tiles, prefix + block * m, both ending in the delimiter, so that no record crosses a copy.  The oracle
runs on the prefix and up to three copies of the block; the answer for the whole text is its records up to the end of
the first copy, then those of the second copy shifted by one block (offsets) and by the block's record closes
(ordinals) for every further copy.  That prediction is checked against the oracle on three copies before it is used."""
import ctypes
import random
import pytest
import _oracle, _corpus
import agrep_b200 as ag
from agrep_b200 import _lib, shard

pytestmark = pytest.mark.gpu

MiB = 1 << 20
SENTINEL = -0x5A5A5A5A5A5A5A5B         # no record field takes this value
FILL = "dfgijklmnopqrtvwxyz"           # no letter of "because each": filler holds none of its anchors
DEV = "cuda"


# ---- texts ----------------------------------------------------------------------------------
def filler(rnd, length):
    """filler lines of `length` bytes in all, each ending in '\\n'"""
    assert length != 1
    out = []
    while length:
        ln = length if length <= 80 else rnd.randint(2, min(80, length - 2))
        out.append("".join(" " if rnd.random() < 0.18 else rnd.choice(FILL) for _ in range(ln - 1)) + "\n")
        length -= ln
    return "".join(out).encode()


def planted_block(rnd, size, lines, n_plants):
    """`size` bytes of filler lines with n_plants lines drawn from `lines`, each starting at a 64-byte boundary.
    Returns (block, start offsets of the planted lines)."""
    slots = sorted(rnd.sample(range(1, size // 64 - 1), n_plants))
    out, at, starts = [], 0, []
    for s in slots:
        ln = rnd.choice(lines)
        assert len(ln) <= 48
        out.append(filler(rnd, s * 64 - at))
        out.append(ln)
        starts.append(s * 64)
        at = s * 64 + len(ln)
    out.append(filler(rnd, size - at))
    block = b"".join(out)
    assert len(block) == size
    return block, starts


# ---- the tiled oracle -----------------------------------------------------------------------
def oracle_rows(pattern, levels=False, **kw):
    """text -> (count, [(begin, end, ordinal[, level]), ...]) by the oracle"""
    a = _oracle.compile(pattern, **kw)
    if levels:
        return lambda text: (lambda cnt, hist, recs: (cnt, recs))(*_oracle.scan_levels(a, kw["k"], text))
    return lambda text: _oracle.scan(a, text)


def oracle_count(pattern, **kw):
    a = _oracle.compile(pattern, **kw)
    return lambda text: (_oracle.scan(a, text, want_records=False)[0], [])


class Tiles:
    """prefix + block * m, and what the oracle says about it, from the prefix and up to three copies of the block"""

    def __init__(self, prefix, block, m, delim=b"\n"):
        assert m >= 2 and prefix.endswith(delim[-1:]) and block.endswith(delim[-1:])
        self.prefix, self.block, self.m, self.delim = prefix, block, m, delim
        self.n = len(prefix) + m * len(block)
        base = shard.count_closes(b"", delim)
        self.block_closes = shard.count_closes(block, delim) - base
        first = shard.count_closes(prefix + block, delim)
        assert shard.count_closes(prefix + block * 3, delim) == first + 2 * self.block_closes
        self.n_closes = first + (m - 1) * self.block_closes

    def host(self):
        return self.prefix + self.block * self.m

    def device(self):
        """the text in HBM (16-byte aligned, 64 zero bytes behind it), built there from one copy of the block"""
        import torch
        t = torch.zeros(self.n + 64, dtype=torch.uint8, device=DEV)
        p, b = len(self.prefix), len(self.block)
        t[:p] = torch.frombuffer(bytearray(self.prefix), dtype=torch.uint8).to(DEV)
        t[p:self.n].view(self.m, b).copy_(torch.frombuffer(bytearray(self.block), dtype=torch.uint8).to(DEV).expand(self.m, b))
        return t

    def expect(self, scan):
        """scan: text -> (count, rows), rows (begin, end, ordinal, ...).  Returns the count over the whole text and its
        rows as an int64 tensor on the device (None for a count-only scan)."""
        import torch
        h, head = scan(self.prefix + self.block)
        c2, two = scan(self.prefix + self.block * 2)
        c3, three = scan(self.prefix + self.block * 3)
        t, tail = c2 - h, two[h:]
        assert two[:h] == head
        step = lambda r: (r[0] + len(self.block), r[1] + len(self.block), r[2] + self.block_closes) + tuple(r[3:])
        assert c3 == h + 2 * t and three == head + tail + [step(r) for r in tail], "the tiled construction does not hold"
        count = h + (self.m - 1) * t
        if not head and not tail:
            return count, None
        ncol = len((head or tail)[0])
        H = torch.tensor(head, dtype=torch.int64).reshape(-1, ncol).to(DEV)
        T = torch.tensor(tail, dtype=torch.int64).reshape(-1, ncol).to(DEV)
        inc = torch.tensor([len(self.block), len(self.block), self.block_closes] + [0] * (ncol - 3), dtype=torch.int64, device=DEV)
        copies = torch.arange(self.m - 1, dtype=torch.int64, device=DEV).view(-1, 1, 1) * inc
        rows = torch.cat([H, (T.unsqueeze(0) + copies).reshape(-1, ncol)])
        assert rows.shape[0] == count
        return count, rows


# ---- calls ----------------------------------------------------------------------------------
def records_buffer(capacity):
    """records tensor of capacity + 64 rows, every row the sentinel"""
    import torch
    return torch.full((capacity + 64, 4), SENTINEL, dtype=torch.int64, device=DEV)


def host_scan(p, ptr, n, want, capacity):
    """agb_scan_host into a host tensor of capacity rows (no retry, no Python list of the records)"""
    import torch
    recs = torch.empty((max(capacity, 1), 4), dtype=torch.int64)
    res = _lib.Result()
    rc = _lib.lib().agb_scan_host(p._h, ctypes.c_void_p(ptr), n, want, ctypes.c_void_p(recs.data_ptr()), capacity, ctypes.byref(res))
    assert rc == 0, _lib.lib().agb_last_error()
    return res, recs


def first_list_size(n):
    """the candidate list a first scan of n bytes gets (scan.cu records_launch + ws_cand_reserve, no size hint yet)"""
    w = max(1 << 20, (n + 15) // 16 // 512 + 65536)
    return w + w // 4


def every_byte_threshold(n):
    """more survivors than this and the record stage walks every byte instead of a list (scan.cu stages_after_front)"""
    return (n + 15) // 16 // 20 + 1024


# ---- 1. the candidate list overflows and the record stage runs again --------------------------
PATTERN = "because each"


def dense_tiles():
    """64 MiB in which nearly every line matches 'because each' at k = 2: more survivors than the first list holds
    and than the list form takes"""
    rnd = random.Random(101)
    lines, size = [], 0
    while size < 65536 - 64:
        if rnd.random() < 0.05:
            ln = filler(rnd, rnd.randint(8, 30))
        else:
            ln = (rnd.choice(["", "dk ", "zq "]) + _corpus.mutate(rnd, PATTERN, rnd.randint(0, 2)) + rnd.choice(["", " fm", " y"]) + "\n").encode()
        lines.append(ln)
        size += len(ln)
    block = b"".join(lines) + filler(rnd, 65536 - size)
    prefix = filler(rnd, 200) + b"because each\n"
    return Tiles(prefix, block, 1024)


def sparse_tiles():
    """512 MiB with one exact 'because each' per 356 bytes, each at a 16-byte boundary: every one of them leaves
    exactly one surviving chunk after stage 1.5, 23 per 8 KiB block -- more than the first list holds, fewer than
    the every-byte forms are taken for"""
    rnd = random.Random(102)
    block, _ = planted_block(rnd, 8192, [b"because each\n"], 23)
    prefix, _ = planted_block(rnd, 320, [b"because each\n"], 2)
    return Tiles(prefix, block, 65536)


@pytest.mark.parametrize("branch", ["dense", "sparse"])
def test_candidate_list_rerun(branch):
    """A first scan sizes the candidate list without knowing the survivors; when they do not fit, the record stage runs
    again -- with the list sized from the count (sparse) or over every byte (dense).  The list with ordinals, the
    number of record closes, the count, the -c -v count and (dense) the streamed entry, each on a fresh workspace,
    against the tiled oracle."""
    import torch
    L = _lib.lib()
    tiles = dense_tiles() if branch == "dense" else sparse_tiles()
    n, n_chunks = tiles.n, (tiles.n + 15) // 16
    kw = dict(k=2, linenum=1)
    count, rows = tiles.expect(oracle_rows(PATTERN, **kw))
    inv_count, _ = tiles.expect(oracle_count(PATTERN, inverse=1, **kw))
    text = tiles.device()
    p = ag.Pattern(PATTERN, **kw)
    first, threshold = first_list_size(n), every_byte_threshold(n)

    def with_list():
        recs = records_buffer(count)
        res = p.scan_device(text.data_ptr(), n, d_records=recs.data_ptr(), capacity=count + 64, ordinals=True)
        return res, recs

    L.agb_shutdown()
    l0 = L.agb_kernel_launches()
    r1, recs1 = with_list()
    l1 = L.agb_kernel_launches()
    r2, recs2 = with_list()                      # the same again: the list is sized from the first scan's survivors
    l2 = L.agb_kernel_launches()
    # the rerun: the record stage's count, scan and emit launches and the ordinals pass once more (the planner's sample,
    # which a second scan of the same text skips, is a single launch)
    assert (l1 - l0) > (l2 - l1) + 2, (l1 - l0, l2 - l1)
    if branch == "dense":
        assert r1.n_flagged == n_chunks                          # every-byte form: all chunks
        assert r2.n_flagged > threshold                          # (list form this time: the survivors)
    else:
        assert first < r1.n_flagged <= threshold, (first, r1.n_flagged, threshold)
        assert r2.n_flagged == r1.n_flagged
    for res, recs in ((r1, recs1), (r2, recs2)):
        assert res.n_matched == count and res.n_records == count and not res.truncated
        assert res.n_closes == tiles.n_closes, (res.n_closes, tiles.n_closes)
        assert torch.equal(recs[:count, :3], rows)
        assert bool((recs[count:] == SENTINEL).all())
    del recs1, recs2

    L.agb_shutdown()
    rc = p.scan_device(text.data_ptr(), n)
    assert rc.n_matched == count
    assert rc.n_flagged == r1.n_flagged

    # agrep -c -v: records minus matching records, the records from the close count of the positive scan
    L.agb_shutdown()
    ri = ag.Pattern(PATTERN, inverse=1, **kw).scan_device(text.data_ptr(), n)
    assert ri.n_flagged == r1.n_flagged                           # the complement path, after the same rerun
    assert ri.n_matched == inv_count, (ri.n_matched, inv_count)

    if branch == "dense":
        del text
        hb = torch.frombuffer(bytearray(tiles.host()), dtype=torch.uint8)
        L.agb_shutdown()
        rh, recs = host_scan(p, hb.data_ptr(), n, _lib.WANT_RECORDS | _lib.WANT_ORDINALS, count + 64)
        assert rh.n_flagged == n_chunks
        assert rh.n_matched == count and rh.n_records == count and rh.n_closes == tiles.n_closes, (rh.n_matched, rh.n_closes, tiles.n_closes)
        assert torch.equal(recs[:count, :3], rows.cpu())
    L.agb_shutdown()


# ---- 2. lists cut short by the capacity --------------------------------------------------------
def _two_per_chunk():
    rnd = random.Random(201)
    return planted_block(rnd, 1 << 16, [b"because\nbecause\n"], 300)[0]


def _equal_anchors():
    rnd = random.Random(202)
    return planted_block(rnd, 1 << 17, [b"abababab\n", b"dd ababxbab k\n", b"abaabab\n", b"abababab abababab\n"], 600)[0]


TRUNC_CASES = {
    # name: (pattern, options, text, levels)
    "list_refined": ("because each", dict(k=2, linenum=1),
                     lambda: ag.corpus_host(1 << 20, needle="because each", needle_every=1, needle_maxedits=3), True),
    "list_unrefined": ("abababab", dict(k=1, linenum=1), _equal_anchors, True),
    "list_several_per_chunk": ("because", dict(k=1, linenum=1), _two_per_chunk, True),
    "slices_class": ("t[a-z]e", dict(k=0, linenum=1), lambda: _corpus.make_text(400, seed=51), False),
    "slices_inverse": ("because", dict(k=1, linenum=1, inverse=1), lambda: _corpus.make_text(400, seed=52), False),
    "dense_wildcard": ("gover#ent", dict(k=1, linenum=1, inverse=1), lambda: _corpus.make_text(400, seed=53), False),
    "dense_run_delim": ("t[hx]e", dict(k=1, linenum=1, delim="$$"), lambda: _corpus.make_text(1200, seed=54, paragraphs=True), True),
}


def _assert_form(name, d, res, n):
    n_chunks = (n + 15) // 16
    anchors = [d.anchor[i] for i in range(d.n_anchors)]
    if name.startswith("list"):
        assert d.plan == _lib.PLAN_ANCHORS and 0 < res.n_flagged <= every_byte_threshold(n), (name, res.n_flagged)
        if name == "list_unrefined":
            assert len(anchors) == 2 and anchors[0] == anchors[1]     # equal anchors at different offsets: no stage 1.5
        else:
            assert d.refine and len(set(anchors)) == len(anchors)
    else:
        assert d.plan == _lib.PLAN_ALL and res.n_flagged == n_chunks, (name, res.n_flagged)
        if name.startswith("slices"):
            assert d.wildmask == 0 and d.L == 1
        else:
            assert d.wildmask != 0 or (d.L > 1 and d.delim_kind != 0)


@pytest.mark.parametrize("name", sorted(TRUNC_CASES))
def test_truncated_lists(name):
    """capacity below, at and above the number of records: exactly the first min(n, capacity) records of the oracle's
    list (with ordinals, and levels where asked) are written and nothing after them; n_records, truncated, n_matched and
    n_closes as for the whole list.  Through agb_scan_device and agb_scan_host with an explicit capacity."""
    import torch
    pattern, kw, make, levels = TRUNC_CASES[name]
    data = make()
    n = len(data)
    cnt, recs = oracle_rows(pattern, levels=levels, **kw)(data)
    assert cnt >= 100, (name, cnt)
    want = torch.tensor(recs, dtype=torch.int64).to(DEV)
    closes = shard.count_closes(data, kw.get("delim", "\n").replace("$$", "\n\n").encode())
    caps = [1, cnt - 1, cnt, cnt + 1]
    if name == "list_several_per_chunk":
        # a cut between two records that close in the same 16-byte chunk: both belong to one candidate
        pairs = [i for i in range(cnt - 1) if recs[i][1] // 16 == recs[i + 1][1] // 16]
        assert len(pairs) > 100
        caps.append(pairs[len(pairs) // 2] + 1)
    p = ag.Pattern(pattern, **kw)
    text = torch.frombuffer(bytearray(data + b"\0" * 64), dtype=torch.uint8).to(DEV)
    for cap in caps:
        k = min(cnt, cap)
        buf = records_buffer(cap)
        res = p.scan_device(text.data_ptr(), n, d_records=buf.data_ptr(), capacity=cap, levels=levels, ordinals=True)
        _assert_form(name, p.desc, res, n)
        assert (res.n_matched, res.n_records, res.truncated, res.n_closes) == (cnt, k, int(cnt > cap), closes), (name, cap)
        assert torch.equal(buf[:k, :3], want[:k, :3]), (name, cap)
        if levels:
            assert torch.equal(buf.view(torch.int32)[:k, 6].to(torch.int64), want[:k, 3]), (name, cap)
        assert bool((buf[k:] == SENTINEL).all()), (name, cap)
        rh, got = p.scan_host(data, capacity=cap, levels=levels, ordinals=True)
        assert (rh.n_matched, rh.n_records, rh.truncated, rh.n_closes) == (cnt, k, int(cnt > cap), closes), (name, cap)
        cols = 4 if levels else 3
        assert [g[:cols] for g in got] == [tuple(r[:cols]) for r in recs[:k]], (name, cap)


# ---- 3. -B lists on one device -----------------------------------------------------------------
def test_bestmatch_lists():
    """-B with a record list: no exact match, more than 1024 records at level 1 with level-2 records among them.  A list
    with room for every level-2 record is filtered to level 1 in place (one CTA over several tiles, order kept); one that
    holds the level-1 records only comes from a rescan at level 1; a smaller one is a prefix of that."""
    import torch
    L = _lib.lib()
    rnd = random.Random(301)
    lvl1 = [b"becase each\n", b"dd because eaxh k\n", b"bxcause each\n", b"because ach\n"]
    lvl2 = [b"bcase each\n", b"becaue eah\n"]
    block, _ = planted_block(rnd, 4096, lvl1 * 3 + lvl2, 40)
    tiles = Tiles(filler(rnd, 130) + b"because eac\n", block, 96)
    total, rows = tiles.expect(oracle_rows(PATTERN, levels=True, k=2, linenum=1))
    lv = rows[:, 3]
    best_rows = rows[lv == 1]
    n_best = best_rows.shape[0]
    assert int((lv == 0).sum()) == 0 and n_best > 1024 and total - n_best > 100
    text = tiles.device()
    deltas = {}
    for what, cap in (("filter", total + 16), ("rescan", (n_best + total) // 2), ("prefix", n_best // 3)):
        buf = records_buffer(cap)
        l0 = L.agb_kernel_launches()
        best, res = ag.bestmatch_device(PATTERN, text.data_ptr(), tiles.n, d_records=buf.data_ptr(), capacity=cap)
        deltas[what] = L.agb_kernel_launches() - l0
        k = min(n_best, cap)
        assert (best, res.n_matched, res.n_records, res.truncated) == (1, n_best, k, int(n_best > cap)), what
        assert torch.equal(buf[:k, :2], best_rows[:k, :2]), what
        assert bool((buf.view(torch.int32)[:k, 6] == 1).all()), what
        assert bool((buf[cap:] == SENTINEL).all()), what
    assert deltas["rescan"] > deltas["filter"] and deltas["prefix"] > deltas["filter"], deltas   # a second scan, not the filter


# ---- 4. the streamed entry across its 64 MiB slices -------------------------------------------
H2D_SLICE = 64 * MiB


def _newline_block():
    rnd = random.Random(401)
    return planted_block(rnd, 4096, [b"because each\n", b"dd becase each k\n", b"because eaxh\n"], 6)


def _paragraph_block():
    """4 KiB of paragraphs separated by '\\n\\n', one separator a run of four newlines; returns (block, run start)"""
    rnd = random.Random(402)
    out, run = [], None
    for i in range(10000):
        if sum(map(len, out)) >= 3600:
            break
        para = [filler(rnd, rnd.randint(20, 70))[:-1] for _ in range(rnd.randint(1, 4))]
        if rnd.random() < 0.4:
            para.insert(rnd.randrange(len(para) + 1), b"xx because eah y")
        out.append(b"\n".join(para))
        if i == 6:
            run = sum(map(len, out))
            out.append(b"\n\n\n\n")
        else:
            out.append(b"\n\n")
    used = sum(map(len, out))
    out.append(filler(rnd, 4096 - used - 1)[:-1] + b"\n\n")
    block = b"".join(out)
    assert len(block) == 4096 and block[run:run + 4] == b"\n\n\n\n" and block[run + 4:run + 5] != b"\n"
    return block, run


def _slice_case(name):
    """(block, position in the block on which every slice boundary falls, delimiter)"""
    if name == "dollar_run":
        block, run = _paragraph_block()
        return block, run + 2, "$$"
    block, starts = _newline_block()
    a = block.index(b"beca", starts[0])          # the first anchor of the first matching line
    if name == "newline":
        return block, block.index(b"\n", a), None
    return block, a + int(name[len("anchor"):]), None


SLICE_CASES = ["anchor%+d" % d for d in range(-3, 4)] + ["newline", "dollar_run"]


@pytest.mark.parametrize("name", SLICE_CASES)
def test_streamed_slice_edges(name):
    """agb_scan_host moves the text in 64 MiB slices and runs stage 1 per slice (the last chunk of a slice reads 4 bytes
    into the next; with -n the delimiters are counted per slice there too).  About three slices, each boundary on a
    chosen byte: around the first anchor of a matching line, on the newline that closes it, inside a '$$' run.  List
    with ordinals, count and record closes, from pageable and page-locked memory, against the tiled oracle and against
    agb_scan_device on the same bytes."""
    import torch
    rnd = random.Random(403)
    block, at, delim = _slice_case(name)
    pre = (-at) % len(block)
    if pre < 3:
        pre += len(block)
    dl = b"\n\n" if delim else b"\n"
    tiles = Tiles(filler(rnd, pre - 1) + b"\n", block, (2 * H2D_SLICE + 8 * MiB) // len(block), delim=dl)
    n = tiles.n
    for boundary in (H2D_SLICE, 2 * H2D_SLICE):
        assert (boundary - pre) % len(block) == at
    kw = dict(k=2, linenum=1)
    if delim:
        kw["delim"] = delim
    count, rows = tiles.expect(oracle_rows(PATTERN, **kw))
    assert count > 1000
    p = ag.Pattern(PATTERN, **kw)
    want = _lib.WANT_RECORDS | _lib.WANT_ORDINALS
    cap = count + 64
    hb = torch.frombuffer(bytearray(tiles.host()), dtype=torch.uint8)
    rows_h = rows.cpu()

    dev = torch.zeros(n + 64, dtype=torch.uint8, device=DEV)
    dev[:n].copy_(hb)
    buf = records_buffer(count)
    rd = p.scan_device(dev.data_ptr(), n, d_records=buf.data_ptr(), capacity=cap, ordinals=True)
    assert (rd.n_matched, rd.n_records, rd.n_closes) == (count, count, tiles.n_closes), (name, rd.n_matched, rd.n_closes)
    assert torch.equal(buf[:count, :3], rows)
    del dev, buf

    pinned = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    pinned.copy_(hb)
    for src in (hb, pinned):
        res, recs = host_scan(p, src.data_ptr(), n, want, cap)
        assert (res.n_matched, res.n_records, res.n_closes) == (count, count, tiles.n_closes), (name, res.n_matched, res.n_closes)
        assert torch.equal(recs[:count, :3], rows_h), name
        rc, _ = host_scan(p, src.data_ptr(), n, _lib.WANT_COUNT, 0)
        assert rc.n_matched == count, name
