"""The KV page allocator (fastllm_b200/csrc/kv_pool.hpp), checked on the CPU: tests/kv_pool_driver.cpp compiles the header into a host
program that replays a command script and prints the allocator's state after every command.  Covered: the home-first, then
lowest-free policy; reference counts through forks, forks of forks and resets of a forked source; that only full pages are shared;
that a reservation or fork the pool cannot cover changes nothing; and that the default pool keeps the identity table -- without a
single table update -- for the uniform, slot and packed call patterns of the existing tests."""
import json
import os
import random
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAGE = 64


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("kv_pool") / "kv_pool_driver")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.run([nvcc, "-std=c++17", "-O1", os.path.join(ROOT, "tests", "kv_pool_driver.cpp"), "-o", exe], check=True,
                   capture_output=True)
    return exe


def run(exe, cmds):
    out = subprocess.run([exe], input="\n".join(cmds) + "\n", check=True, capture_output=True, text=True).stdout
    return [json.loads(line) for line in out.splitlines()]


def pages_for(tokens):
    return -(-tokens // PAGE)


class RefPool:
    """The allocation policy written out directly: what every command must leave behind."""

    def __init__(self, b, p, n):
        self.b, self.p, self.n = b, p, n
        self.ref = [0] * n
        self.pages = [[] for _ in range(b)]

    def unassigned(self, s, p):
        return s * self.p + p if s * self.p + p < self.n else 0

    def table(self):
        return [self.pages[s][p] if p < len(self.pages[s]) else self.unassigned(s, p) for s in range(self.b) for p in range(self.p)]

    def free(self):
        return sum(r == 0 for r in self.ref)

    def take(self, s):
        home = s * self.p + len(self.pages[s])
        page = home if home < self.n and self.ref[home] == 0 else self.ref.index(0)
        self.ref[page] = 1
        self.pages[s].append(page)
        return page

    def reserve(self, req):
        if sum(max(0, pages_for(t) - len(self.pages[s])) for s, t in req) > self.free():
            return False
        for s, t in sorted(req):
            while len(self.pages[s]) < pages_for(t):
                self.take(s)
        return True

    def release(self, s):
        for pg in self.pages[s]:
            self.ref[pg] -= 1
        self.pages[s] = []

    def fork(self, src, dst, n):
        full, partial = n // PAGE, n % PAGE != 0
        if src == dst or self.pages[dst] or len(self.pages[src]) < pages_for(n) or (partial and self.free() == 0):
            return False, [-1, -1]
        for pg in self.pages[src][:full]:
            self.ref[pg] += 1
            self.pages[dst].append(pg)
        return True, ([self.pages[src][full], self.take(dst)] if partial else [-1, -1])


def replay(exe, b, p, n, script):
    """Runs script (commands as tuples) on the driver and on RefPool; every state must agree, and every flush must list exactly the
    table entries that changed."""
    ref = RefPool(b, p, n)
    cmds = [f"init {b} {p} {n}"] + [" ".join(map(str, c)) for c in script]
    states = run(exe, cmds)
    prev = ref.table()
    assert states[0]["table"] == prev and states[0]["flush"] == []
    for cmd, st in zip(script, states[1:]):
        op = cmd[0]
        ok, copy = True, [-1, -1]
        if op == "reserve":
            ok = ref.reserve(list(zip(cmd[1::2], cmd[2::2])))
        elif op == "release":
            ref.release(cmd[1])
        elif op == "release_all":
            for s in range(b):
                ref.release(s)
        elif op == "fork":
            ok, copy = ref.fork(*cmd[1:])
        assert (bool(st["ok"]), st["copy"]) == (ok, copy), cmd
        assert st["ref"] == ref.ref and st["pages"] == ref.pages and st["free"] == ref.free() and st["total"] == n, cmd
        table = ref.table()
        assert st["table"] == table, cmd
        assert st["flush"] == [[i, table[i]] for i in range(len(table)) if table[i] != prev[i]], cmd
        prev = table
    return states[1:]


def test_home_page_first_then_lowest_free(driver):
    # 4 slots x 4 pages of table, a pool of 6 pages: slot 0's and slot 1's home pages exist (0-3, 4-5), slots 2-3 have none
    st = replay(driver, 4, 4, 6, [("reserve", 2, 100), ("reserve", 0, 64), ("reserve", 1, 1), ("reserve", 0, 130),
                                  ("release", 2), ("reserve", 3, 65)])
    assert st[0]["pages"][2] == [0, 1]            # no home pages: the lowest free ones
    assert st[1]["pages"][0] == [2]               # home page 0 is taken: the lowest free
    assert st[2]["pages"][1] == [4]               # its home page
    assert st[3]["pages"][0] == [2, 3, 5]         # home pages 1 (slot 2) and 2 (itself) are taken: the lowest free ones
    assert st[3]["free"] == 0
    assert st[5]["pages"][3] == [0, 1]


def test_refcounts_through_forks_and_source_reset(driver):
    st = replay(driver, 4, 4, 16, [("reserve", 0, 150), ("fork", 0, 1, 150), ("reserve", 1, 151), ("fork", 1, 2, 151),
                                   ("fork", 2, 3, 128), ("release", 0), ("reserve", 2, 200), ("release", 1), ("release", 2),
                                   ("release", 3)])
    src = st[0]["pages"][0]
    assert src == [0, 1, 2]
    assert st[1]["pages"][1][:2] == src[:2] and st[1]["pages"][1][2] != src[2]      # full pages shared, the partial one copied
    assert st[1]["copy"] == [src[2], st[1]["pages"][1][2]]
    assert [st[1]["ref"][pg] for pg in src] == [2, 2, 1]
    assert [st[3]["ref"][pg] for pg in src[:2]] == [3, 3]                            # fork of a fork
    assert st[4]["copy"] == [-1, -1] and [st[4]["ref"][pg] for pg in src[:2]] == [4, 4]    # a multiple of 64: nothing copied
    assert st[4]["ref"][st[3]["pages"][2][2]] == 1
    assert [st[5]["ref"][pg] for pg in src[:2]] == [3, 3] and st[5]["ref"][src[2]] == 0   # the source's reset keeps shared pages
    assert st[-1]["free"] == 16 and all(r == 0 for r in st[-1]["ref"])


def test_exhausted_reservation_and_fork_change_nothing(driver):
    st = replay(driver, 3, 4, 5, [("reserve", 0, 129), ("reserve", 1, 64, 2, 65), ("reserve", 1, 64, 2, 64),
                                  ("fork", 0, 2, 129), ("fork", 0, 1, 128), ("fork", 1, 1, 10), ("release", 0), ("fork", 1, 0, 64)])
    assert st[1]["ok"] == 0 and st[1]["free"] == 2                       # needs 3 pages, 2 free: nothing taken
    assert st[2]["ok"] == 1 and st[2]["free"] == 0
    assert st[3]["ok"] == 0 and st[4]["ok"] == 0                         # dst not empty
    assert st[5]["ok"] == 0                                              # src == dst
    assert st[7]["ok"] == 1 and st[7]["pages"][0] == [4] and st[7]["ref"][4] == 2
    for a, b in zip(st, st[1:]):
        if not b["ok"]:
            assert (a["ref"], a["pages"], a["table"]) == (b["ref"], b["pages"], b["table"]) and b["flush"] == []


def test_partial_copy_needs_a_free_page(driver):
    st = replay(driver, 2, 2, 2, [("reserve", 0, 100), ("fork", 0, 1, 100), ("fork", 0, 1, 64)])
    assert st[1]["ok"] == 0 and st[1]["flush"] == []      # a partial last page and no free page
    assert st[2]["ok"] == 1 and st[2]["pages"][1] == [0] and st[2]["ref"] == [2, 1]   # full pages only: no free page needed


@pytest.mark.parametrize("b,p", [(1, 4), (3, 2), (8, 5)])
def test_default_pool_keeps_the_identity_table(driver, b, p):
    """fl_cache_create's pool (max_batch * pages_per_seq pages) without forks: every page taken is a home page, the table stays the
    identity and no call ever has a table entry to write (so no call launches anything extra)."""
    rs = random.Random(b * 100 + p)
    cap = p * PAGE
    script, lens = [], [0] * b
    # uniform calls: slots 0..k-1 grow together (prefill, then decode steps across page boundaries), then a reset
    kv = 0
    for t in [3, 1, 61, 1, 1, 64]:
        if kv + t <= cap:
            kv += t
            script.append(("reserve", *[x for s in range(b) for x in (s, kv)]))
    script.append(("release_all",))
    # slot and packed calls: slots of their own lengths, finished slots reset and re-admitted
    for _ in range(40):
        n = rs.randint(1, b)
        slots = rs.sample(range(b), n)
        req = []
        for s in slots:
            add = rs.choice([1, 1, rs.randint(1, PAGE * 2)])
            if lens[s] + add > cap:
                script.append(("release", s))
                lens[s] = 0
            lens[s] += add
            req += [s, lens[s]]
        script.append(("reserve", *req))
    st = replay(driver, b, p, b * p, script)
    ident = list(range(b * p))
    for s in st:
        assert s["ok"] == 1 and s["table"] == ident and s["flush"] == []


def test_random_scripts_match_the_policy(driver):
    """Random reservations, releases and forks on pools smaller than max_batch * pages_per_seq: every state equals the policy's."""
    for seed in range(6):
        rs = random.Random(seed)
        b, p = rs.randint(2, 6), rs.randint(1, 5)
        n = rs.randint(1, b * p)
        script = []
        for _ in range(60):
            op = rs.random()
            if op < 0.55:
                slots = rs.sample(range(b), rs.randint(1, b))
                req = []
                for s in slots:
                    req += [s, rs.randint(1, p * PAGE)]
                script.append(("reserve", *req))
            elif op < 0.75:
                script.append(("release", rs.randrange(b)))
            elif op < 0.8:
                script.append(("release_all",))
            else:
                script.append(("fork", rs.randrange(b), rs.randrange(b), rs.randint(1, p * PAGE)))
        replay(driver, b, p, n, script)
