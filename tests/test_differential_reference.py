"""Differential test against the REAL reference: seeded random DSL pipelines run through Refefer/Dampr's own
MTRunner and through this engine's runner (on the numpy stand-in for the device, tests/fake_device.py) must
give the same multiset of results. This pins the DSL semantics of the host layer — stage fusion, keyed
records, combiners, joins — to the reference itself rather than to a restatement.

The reference's results on the seeded inputs are stored in tests/golden/differential_reference.json.gz. To record
them again from a checkout of the reference (after a change to a pipeline or an input):

    DAMPR_REFERENCE=<checkout of Refefer/Dampr> python -m pytest tests/test_differential_reference.py
"""
import gzip
import os
import random
import subprocess
import sys
import json
import tempfile

import pytest

REF = os.environ.get("DAMPR_REFERENCE")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "differential_reference.json.gz")


def reference(case, driver, *args):
    """The last stdout line of `python -c driver <reference checkout> *args`, parsed as JSON: the stored result for
    `case`, or, when DAMPR_REFERENCE names a checkout, the result of running the reference now, which is stored."""
    with gzip.open(GOLDEN, "rt") as f:
        stored = json.load(f)
    if not REF:
        return stored[case]
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)   # the reference's `dampr` package, not this repository's shim
    p = subprocess.run([sys.executable, "-c", driver, REF] + list(args), capture_output=True, text=True, env=env,
                       cwd=tempfile.gettempdir(), timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    stored[case] = json.loads(p.stdout.strip().split("\n")[-1])
    with open(GOLDEN, "wb") as f:
        f.write(gzip.compress(json.dumps(stored, sort_keys=True, separators=(",", ":")).encode(), mtime=0))
    return stored[case]


def pipelines(seed, n_cases):
    """Source text of n_cases pipelines over `Dampr` and an input list `items` (evaluated in both engines)."""
    rng = random.Random(seed)
    out = []
    for _ in range(n_cases):
        m = rng.choice([3, 5, 7, 11])
        k = rng.randint(1, 4)
        c = rng.randint(-3, 3)
        base = "Dampr.memory(items, partitions=%d)" % rng.choice([1, 2, 5])
        steps = []
        for _j in range(rng.randint(0, 2)):
            steps.append(rng.choice([
                ".map(lambda x: x * %d + %d)" % (k, c),
                ".filter(lambda x: x %% %d != %d)" % (m, rng.randrange(m)),
                ".flat_map(lambda x: [x, x + %d])" % k,
            ]))
        tail = rng.choice([
            ".group_by(lambda x: x %% %d).reduce(lambda k, it: sum(it))" % m,
            ".group_by(lambda x: x %% %d, lambda x: x * 2).reduce(lambda k, it: len(list(it)))" % m,
            ".a_group_by(lambda x: x %% %d).sum()" % m,
            ".a_group_by(lambda x: x %% %d, lambda x: 1).reduce(lambda a, b: a + b)" % m,
            ".count(lambda x: x %% %d)" % m,
            ".fold_by(lambda x: x %% %d, max)" % m,
            ".fold_by(lambda x: x %% %d, min, lambda x: -x)" % m,
            ".mean(lambda x: x %% %d, lambda x: x)" % m,
            ".sort_by(lambda x: (x %% %d, x))" % m,
            ".map(lambda x: (x %% %d, x)).map_values(lambda v: v + 1).map_keys(lambda q: q * 2)" % m,
            ".group_by(lambda x: x %% %d).reduce(lambda k, it: sum(it)).join(" % m + base +
            ".group_by(lambda x: x %% %d).reduce(lambda k, it: max(it))).reduce(lambda l, r: (list(l), list(r)))" % m,
            ".len()",
            ".topk(%d)" % rng.randint(1, 5),
            ".cross_right(" + base + ".len(), lambda x, t: x * 1000 + t)",
        ])
        out.append(base + "".join(steps) + tail)
    return out


DRIVER = r"""
import sys, json
sys.path.insert(0, sys.argv[1])
from dampr import Dampr
items = json.loads(sys.argv[2])
res = []
for src in json.loads(sys.argv[3]):
    r = list(eval(src).run())
    res.append(sorted(repr(x) for x in r))
print(json.dumps(res))
"""


def test_random_pipelines_agree_with_the_reference(monkeypatch):
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    rng = random.Random(7)
    items = [rng.randint(-50, 200) for _ in range(300)]
    srcs = pipelines(2024, 60)
    # the reference runs in its own interpreter (its `dampr` package would shadow the shim here)
    ref = reference("random_pipelines", DRIVER, json.dumps(items), json.dumps(srcs))
    monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
    monkeypatch.setattr(plan, "_BUFFERS", {})
    for src, exp in zip(srcs, ref):
        got = sorted(repr(x) for x in eval(src, {"Dampr": Dampr, "items": items}).run())
        if ".mean(" in src:
            g = [eval(x) for x in got]
            e = [eval(x) for x in exp]
            assert len(g) == len(e) and all(a[0] == b[0] and abs(a[1] - b[1]) <= 1e-9 * max(1.0, abs(b[1])) for a, b in zip(g, e)), src
        else:
            assert got == exp, src


TEXT_DRIVER = r"""
import sys, json, re, math
sys.path.insert(0, sys.argv[1])
from dampr import Dampr
RX = re.compile(r'[^\w]+')
path = sys.argv[2]
res = []
for src in json.loads(sys.argv[3]):
    r = list(eval(src).run())
    res.append(sorted(repr(x) for x in r))
print(json.dumps(res))
"""


def text_pipelines(seed, n_cases, longest):
    """chunk sizes start above the longest line: below that the reference yields the line that follows an
    over-long line once per chunk the long line spans (SURVEY §8(a) T1), which the parity contract excludes."""
    rng = random.Random(seed)
    out = []
    for _ in range(n_cases):
        chunk = rng.choice([longest + 1, 2 * longest + 3, max(4096, longest + 7), 1 << 20])
        base = "Dampr.text(path, %d)" % chunk
        out.append(base + rng.choice([
            ".flat_map(lambda x: x.split()).count()",
            ".flat_map(lambda x: set(RX.split(x.lower()))).count()",
            ".flat_map(lambda x: RX.split(x.lower())).count()",
            ".len()",
            ".map(lambda x: len(x)).a_group_by(lambda x: x % 5).sum()",
            ".filter(lambda x: len(x) % 2 == 0).map(lambda x: x[:3]).count()",
            ".flat_map(lambda x: x.upper().split()).fold_by(lambda w: w[:1], lambda a, b: a + b, lambda w: 1)",
            ".flat_map(lambda x: x.split()).count().sort_by(lambda wc: (-wc[1], wc[0]))",
            ".flat_map(lambda x: set(RX.split(x.lower()))).count().cross_right(" + base +
            ".len(), lambda df, total: (df[0], df[1], math.log(1 + (float(total) / df[1]))))",
        ]))
    return out


@pytest.mark.parametrize("path_kind", ["host-map", "scan-plumbing"])
def test_random_text_pipelines_agree_with_the_reference(path_kind, monkeypatch, tmp_path):
    """Text inputs with assorted chunk sizes (line ownership at chunk seams, the '' token of re.split,
    str.split) through the reference and through this engine: once with every text stage as a host map, once
    through the lowered path's plumbing (plan.TextScan) with the stand-in tokeniser of tests/fake_device.py."""
    import math
    import re
    from fake_device import FakeCtx
    from oracle import gen
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    RX = re.compile(r"[^\w]+")
    # '\r' and '\r\n' line ends (universal newlines) and UTF-8 text: one chunk per file, because with several
    # chunks the reference's character positions drift from its byte seeks and it yields some lines twice
    cr = b"a b\r\nCcc d_1\r\n\r\nx.y 42\r\n" * 20
    mixed = b"a\rb b\r\nc\n\rd e-e\n" * 15
    utf8 = "na\u00efve caf\u00e9\nplain line\n\u00dcber \u00fcber\n".encode("utf-8") * 10
    for ci, data in enumerate((gen.text(5, 400, V=300), gen.dirty_text(11, 300, 200), b"", b"one line without newline",
                               cr, mixed, utf8)):
        path = str(tmp_path / ("c%d.txt" % ci))
        with open(path, "wb") as f:
            f.write(data)
        longest = max([len(l) + 1 for l in data.split(b"\n")] + [1]) if ci < 4 else len(data) + 1
        srcs = text_pipelines(100 + ci, 14, longest)
        ref = reference("text_pipelines_%d" % ci, TEXT_DRIVER, path, json.dumps(srcs))
        if path_kind == "host-map":
            monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
        else:
            from fake_device import FakeTextCtx, FakePinned
            monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeTextCtx()})
            monkeypatch.setattr(plan, "_pinned_ring", lambda n, b: [FakePinned(b) for _ in range(n)])
        monkeypatch.setattr(plan, "_BUFFERS", {})
        for src, exp in zip(srcs, ref):
            got = sorted(repr(x) for x in eval(src, {"Dampr": Dampr, "path": path, "RX": RX, "math": math}).run())
            assert got == exp, (ci, src)


def more_pipelines(seed, n):
    """joins (inner / left / many), unique, prefix / suffix, map-side joins, checkpoints, partition_map /
    partition_reduce, string / tuple keys, float values. Reducers sort their groups first: the order of the values
    inside a group depends on which of the reference's worker processes finished first. (Keys of mixed types are left out: the reference's
    workers die on the sort's TypeError and its parent then waits forever, SURVEY §5.)"""
    rng=random.Random(seed); out=[]
    for _ in range(n):
        m=rng.choice([3,5,7]); base="Dampr.memory(items, partitions=%d)"%rng.choice([1,2,5]); other="Dampr.memory(items[::2], partitions=2)"
        out.append(rng.choice([
            base+".group_by(lambda x: x %% %d).reduce(lambda k, it: sum(it)).join(%s.group_by(lambda x: x %% %d + 1).reduce(lambda k, it: max(it))).left_reduce(lambda l, r: (list(l), list(r)))"%(m,other,m),
            base+".group_by(lambda x: x %% %d).join(%s.group_by(lambda x: x %% %d)).reduce(lambda l, r: (sorted(l), sorted(r)))"%(m,other,m),
            base+".group_by(lambda x: x %% %d).join(%s.group_by(lambda x: x %% %d)).reduce(lambda l, r: (lambda ll, rr: [a*b for a in ll for b in rr[:2]])(sorted(l), sorted(r)), many=True)"%(m,other,m),
            "Dampr.memory(items, partitions=1).group_by(lambda x: x %% %d).unique(lambda v: v %% 2)"%m,   # (one input partition: with several, which value unique() sees first depends on the reference's worker scheduling)
            base+".prefix(lambda x: x %% %d).suffix(lambda x: x[0] + 1)"%m,
            base+".cross_left(%s.filter(lambda x: x %% 17 == 0), lambda a, b: (a, b))"%other,
            base+".cross_set(%s, lambda b, table: (b, b in table), agg=set)"%other,
            base+".cross_set(%s, lambda b, table: (b, sum(table) %% 7))"%other,
            base+".map(lambda x: x + 1).checkpoint().map(lambda x: x * 2).cached().count(lambda x: x %% %d)"%m,
            base+".a_group_by(lambda x: x %% %d).reduce(lambda a, b: a if a > b else b)"%m,
            base+".partition_map(lambda it: [(1, sum(it))]).partition_reduce(lambda groups: [(k, sum(v)) for k, v in groups])",
            base+".group_by(lambda x: x %% %d).partition_reduce(lambda groups: [(k, len(list(v))) for k, v in groups])"%m,
            base+".map(lambda x: str(x)).group_by(lambda s: s[-1]).reduce(lambda k, it: ''.join(sorted(it))[:20])",
            base+".map(lambda x: (x %% %d, float(x) / 3)).a_group_by(lambda kv: kv[0], lambda kv: kv[1]).reduce(lambda a, b: max(a, b))"%m,
            base+".group_by(lambda x: (x % 2, x % 3)).reduce(lambda k, it: sum(it))",
        ]))
    return out


def test_more_random_pipelines_agree_with_the_reference(monkeypatch):
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    for seed, n_items in ((3, 120), (4, 7), (5, 0)):
        rng = random.Random(seed)
        items = [rng.randint(-50, 200) for _ in range(n_items)]
        srcs = more_pipelines(seed * 17, 40)
        ref = reference("more_pipelines_%d" % seed, DRIVER, json.dumps(items), json.dumps(srcs))
        monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
        monkeypatch.setattr(plan, "_BUFFERS", {})
        for src, exp in zip(srcs, ref):
            got = sorted(repr(x) for x in eval(src, {"Dampr": Dampr, "items": items}).run())
            assert got == exp, (n_items, src)


SINK_DRIVER = r"""
import sys, json, os
sys.path.insert(0, sys.argv[1])
from dampr import Dampr
items = json.loads(sys.argv[2])
res = []
for i, src in enumerate(json.loads(sys.argv[3])):
    out = os.path.join(sys.argv[4], "ref%d" % i)
    eval(src).run()
    lines = []
    for fn in sorted(os.listdir(out)):
        with open(os.path.join(out, fn)) as f:
            lines.extend(l.rstrip("\n") for l in f)
    res.append(sorted(lines))
print(json.dumps(res))
"""


def test_sinks_write_the_lines_the_reference_writes(monkeypatch, tmp_path):
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    rng = random.Random(21)
    items = [rng.randint(-50, 200) for _ in range(150)]
    templates = [
        "Dampr.memory(items, partitions=3).count(lambda x: x % 7).sink_tsv(out)",
        "Dampr.memory(items, partitions=2).map(lambda x: (str(x), x / 7.0, x * 10 ** 18)).sink_tsv(out)",
        "Dampr.memory(items, partitions=2).map(lambda x: ('k%d' % x, [x, x / 3.0], {'a': x})).sink_json(out)",
        "Dampr.memory(items, partitions=4).map(lambda x: 'line %d' % x).sink(out)",
        "Dampr.memory(items, partitions=1).mean(lambda x: x % 3, lambda x: x).sink_tsv(out)",
    ]
    ref = reference("sinks", SINK_DRIVER, json.dumps(items), json.dumps(templates), str(tmp_path))
    monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
    monkeypatch.setattr(plan, "_BUFFERS", {})
    for i, (src, exp) in enumerate(zip(templates, ref)):
        out = str(tmp_path / ("ours%d" % i))
        eval(src, {"Dampr": Dampr, "items": items, "out": out}).run()
        lines = []
        for fn in sorted(os.listdir(out)):
            with open(os.path.join(out, fn)) as f:
                lines.extend(l.rstrip("\n") for l in f)
        assert sorted(lines) == exp, src


def key_type_pipelines():
    """Grouping / folding / sorting / joining on keys of assorted types: strings sharing an 8-byte prefix, ints
    beyond 2^63, floats, -0.0, tuples, bools (True == 1), mixed int / float, bytes, the empty string."""
    keyfs = ["lambda x: 'prefix-shared-%03d' % (x % 40)", "lambda x: 'abcdefgh' + str(x % 9) * (x % 4)", "lambda x: x * 10 ** 18", "lambda x: -(x % 5) * 2 ** 62",
             "lambda x: float(x % 6) / 3", "lambda x: (x % 2) * -0.0", "lambda x: (x % 3, str(x % 4))", "lambda x: (x % 3 == 0)", "lambda x: x % 3 if x % 2 else (x % 3 == 1)",
             "lambda x: ''", "lambda x: 2 ** 63 + (x % 3)", "lambda x: -2 ** 63 + (x % 3)", "lambda x: float(x % 3) if x % 2 else x % 3", "lambda x: (str(x % 3),)", "lambda x: b'k%d' % (x % 5)"]
    tails = [".group_by(%s).reduce(lambda k, it: sum(it))", ".a_group_by(%s).sum()", ".count(%s)", ".fold_by(%s, min)", ".sort_by(%s)",
             ".group_by(%s).reduce(lambda k, it: len(list(it))).join(Dampr.memory(items[::3], partitions=2).group_by(%s).reduce(lambda k, it: sum(it))).reduce(lambda l, r: (list(l), list(r)))"]
    srcs=[]
    for kf in keyfs:
        for t in tails:
            srcs.append("Dampr.memory(items, partitions=3)" + (t % ((kf,) * t.count("%s"))))
    return srcs


def test_key_types_agree_with_the_reference(monkeypatch):
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    rng = random.Random(5)
    items = [rng.randint(-50, 200) for _ in range(90)]
    srcs = key_type_pipelines()
    ref = reference("key_types", DRIVER, json.dumps(items), json.dumps(srcs))
    monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
    monkeypatch.setattr(plan, "_BUFFERS", {})
    for src, exp in zip(srcs, ref):
        got = sorted(repr(x) for x in eval(src, {"Dampr": Dampr, "items": items}).run())
        assert got == exp, src


EXPR_DRIVER = r"""
import sys, json
sys.path.insert(0, sys.argv[1])
from dampr import Dampr
items = json.loads(sys.argv[2]); jpath = sys.argv[4]
print(json.dumps([repr(eval(src)) for src in json.loads(sys.argv[3])]))
"""


def test_inputs_outputs_and_empty_cases_agree_with_the_reference(monkeypatch, tmp_path):
    """Dampr.json inputs, multi-output Dampr.run, read(k), empty inputs through every stage kind, topk, sample(0/1),
    first(), empty sides of inner / left joins."""
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    rng = random.Random(9)
    jpath = str(tmp_path / "j.json")
    with open(jpath, "w") as f:
        for i in range(200):
            f.write(json.dumps({"id": i, "tag": "t%d" % (i % 7), "v": rng.randint(-5, 50), "w": [i, i % 3]}) + "\n")
    items = [rng.randint(-20, 60) for _ in range(80)]
    srcs = [
     "sorted(Dampr.json(jpath).map(lambda d: (d['tag'], d['v'])).a_group_by(lambda kv: kv[0], lambda kv: kv[1]).sum().run())",
     "sorted(Dampr.json(jpath, 512).filter(lambda d: d['v'] > 10).map(lambda d: d['id']).run())",
     "sorted(Dampr.json(jpath).group_by(lambda d: d['w'][1], lambda d: d['v']).reduce(lambda k, it: max(it)).run())",
     "[sorted(x) for x in Dampr.run(Dampr.memory(items).count(lambda x: x % 3), Dampr.memory(items).map(lambda x: x + 1).a_group_by(lambda x: x % 2).sum())]",
     "sorted(Dampr.memory(items, partitions=4).count(lambda x: x % 5).read(2))[:0]",
     "len(Dampr.memory(items, partitions=4).count(lambda x: x % 5).read(2))",
     "sorted(Dampr.memory(items).map(lambda x: x % 4).sort_by(lambda x: x).read())",
     "sorted(Dampr.memory(items).group_by(lambda x: x % 3).reduce(lambda k, it: sum(it)).run().read(1)) [:0]",
     "list(Dampr.memory([]).len().run())",
     "list(Dampr.memory([]).count().run())",
     "list(Dampr.memory([5]).mean().run())",
     "sorted(Dampr.memory(items).a_group_by(lambda x: x % 3).first().run())[:0]",
     "sorted(k for k, v in Dampr.memory(items).a_group_by(lambda x: x % 3).first().run())",
     "sorted(Dampr.memory(items).topk(3, lambda x: -x).run())",
     "sorted(Dampr.memory(items).topk(300).run()) == sorted(items)",
     "sorted(Dampr.memory(items).sample(1.0).run()) == sorted(items)",
     "list(Dampr.memory(items).sample(0.0).run())",
     "sorted(Dampr.memory(items).flat_map(lambda x: []).count().run())",
     "sorted(Dampr.memory(items).filter(lambda x: False).group_by(lambda x: x).reduce(lambda k, it: 1).run())",
     "sorted(Dampr.memory(items).filter(lambda x: False).sort_by(lambda x: x).run())",
     "sorted(Dampr.memory(items).filter(lambda x: False).a_group_by(lambda x: 1).sum().join(Dampr.memory(items).a_group_by(lambda x: 1).sum()).reduce(lambda l, r: 1).run())",
     "sorted(Dampr.memory(items).a_group_by(lambda x: 1).sum().join(Dampr.memory(items).filter(lambda x: False).a_group_by(lambda x: 1).sum()).left_reduce(lambda l, r: (list(l), list(r))).run())",
    ]
    ref = reference("inputs_outputs_and_empty_cases", EXPR_DRIVER, json.dumps(items), json.dumps(srcs), jpath)
    monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
    monkeypatch.setattr(plan, "_BUFFERS", {})
    for src, exp in zip(srcs, ref):
        assert repr(eval(src, {"Dampr": Dampr, "items": items, "jpath": jpath})) == exp, src


RECS_DRIVER = r"""
import sys, json
sys.path.insert(0, sys.argv[1])
from dampr import Dampr
recs = [tuple(r) for r in json.loads(sys.argv[2])]
print(json.dumps([sorted(repr(x) for x in eval(src).run()) for src in json.loads(sys.argv[3])]))
"""


def test_lowered_kv_and_frame_stages_agree_with_the_reference(monkeypatch):
    """Binary (key, value) records through the LOWERED path of this engine — device folds / sorts of the
    columns, then the column-at-a-time frame stages (vexpr) — against the reference running the same lambdas
    record by record over the same tuples."""
    import numpy as np
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    from dampr_b200.inputs import ArrayKVInput
    rng = random.Random(13)
    keys = [rng.randint(-40, 40) for _ in range(4000)]
    vals = [rng.randint(-1000, 1000) for _ in range(4000)]
    heads = [".a_group_by(lambda x: x[0], lambda x: x[1]).sum()", ".count(lambda x: x[0])", ".fold_by(lambda x: x[0], min, lambda x: x[1])", ".fold_by(lambda x: x[1] % 50, max, lambda x: x[0])",
             ".group_by(lambda x: x[0], lambda x: x[1]).reduce(lambda k, it: sum(it))", ".group_by(lambda x: x[0], lambda x: x[1]).reduce(lambda k, it: len(list(it)))"]
    tails = ["", ".map(lambda kv: (kv[0], kv[1] * 3 - kv[0], kv[1] / 7))", ".filter(lambda kv: kv[1] > 0).map_values(lambda v: v // 5)", ".fold_by(lambda kv: kv[0] % 7, lambda x, y: x + y, value=lambda kv: kv[1])",
             ".mean(lambda kv: abs(kv[0]) % 5, lambda kv: kv[1])", ".mean(value=lambda kv: float(kv[1]))", ".sort_by(lambda kv: kv[1] - 2 * kv[0])", ".map(lambda kv: kv[0] * kv[1]).a_group_by(lambda x: 1).sum()",
             ".filter(lambda kv: kv[0] != 0).map(lambda kv: (kv[0], kv[1] % kv[0], kv[1] // kv[0], float(kv[1]) / kv[0]))", ".map(lambda kv: -kv[1]).sort_by(lambda x: x)", ".len()",
             ".fold_by(lambda kv: kv[1] % 3, lambda a, b: a if a < b else b, lambda kv: kv[0])", ".map(lambda kv: (kv[0] < kv[1], kv[0] == 0, abs(kv[1]) >= 10))"]
    srcs_ref=[]; srcs_ours=[]
    for h in heads:
        for t in tails:
            srcs_ref.append("Dampr.memory(recs, partitions=3)"+h+t); srcs_ours.append("Dampr.read_input(ArrayKVInput(K, V))"+h+t)
    ref = reference("lowered_kv_and_frame_stages", RECS_DRIVER, json.dumps(list(zip(keys, vals))), json.dumps(srcs_ref))
    K, V = np.array(keys, dtype=np.int64), np.array(vals, dtype=np.int64)
    lowered = 0
    for so, exp in zip(srcs_ours, ref):
        monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
        monkeypatch.setattr(plan, "_BUFFERS", {})
        got = sorted(repr(x) for x in eval(so, {"Dampr": Dampr, "ArrayKVInput": ArrayKVInput, "K": K, "V": V}).run())
        hows = [h for _s, h, _d in runner_mod.LAST_STATS.stages]
        lowered += any("column-at-a-time" in h or "frame keyed fold" in h or "device sort of frame rows" in h for h in hows)
        if ".mean(" in so:
            g, e = [eval(x) for x in got], [eval(x) for x in exp]
            assert len(g) == len(e) and all(a[0] == b[0] and abs(a[1] - b[1]) <= 1e-9 * max(1.0, abs(b[1])) for a, b in zip(g, e)), so
        else:
            assert got == exp, so
    assert lowered >= 40     # the frame stages really took the lowered path


def test_lowered_cross_and_sink_agree_with_the_reference(monkeypatch, tmp_path):
    """The tf-idf tail — cross_right with the 1-row total (memoised per distinct value) and the native
    sink_tsv — over a lowered count frame, against the reference's files for the same records."""
    import math
    import numpy as np
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    from dampr_b200.inputs import ArrayKVInput
    rng = random.Random(17)
    keys = [int(rng.paretovariate(1.2)) % 500 for _ in range(6000)]
    vals = [rng.randint(0, 9) for _ in range(6000)]
    tail = ".count(lambda x: x[0]).cross_right(%s.len(), lambda df, total: (df[0], df[1], math.log(1 + (float(total) / df[1]))), " \
           "memory=True).sink_tsv(out)"
    ref_src = "Dampr.memory(recs, partitions=3)" + tail % "Dampr.memory(recs, partitions=3)"
    driver = r"""
import sys, json, os, math
sys.path.insert(0, sys.argv[1])
from dampr import Dampr
recs = [tuple(r) for r in json.loads(sys.argv[2])]
out = sys.argv[4]
eval(sys.argv[3]).run()
lines = []
for fn in sorted(os.listdir(out)):
    with open(os.path.join(out, fn)) as f:
        lines.extend(l.rstrip("\n") for l in f)
print(json.dumps(sorted(lines)))
"""
    exp = reference("lowered_cross_and_sink", driver, json.dumps(list(zip(keys, vals))), ref_src, str(tmp_path / "ref"))
    monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
    monkeypatch.setattr(plan, "_BUFFERS", {})
    K, V = np.array(keys, dtype=np.int64), np.array(vals, dtype=np.int64)
    out = str(tmp_path / "ours")
    src = "Dampr.read_input(ArrayKVInput(K, V))" + tail % "Dampr.read_input(ArrayKVInput(K, V))"
    eval(src, {"Dampr": Dampr, "ArrayKVInput": ArrayKVInput, "K": K, "V": V, "math": math, "out": out}).run()
    hows = [h for _s, h, _d in runner_mod.LAST_STATS.stages]
    assert any("memoised per distinct" in h for h in hows) and any("native frame sink" in h for h in hows), hows
    lines = []
    for fn in sorted(os.listdir(out)):
        with open(os.path.join(out, fn)) as f:
            lines.extend(l.rstrip("\n") for l in f)
    assert sorted(lines) == exp


TWO_DRIVER = r"""
import sys, json
sys.path.insert(0, sys.argv[1])
from dampr import Dampr
recs = [tuple(r) for r in json.loads(sys.argv[2])]; recs2 = [tuple(r) for r in json.loads(sys.argv[4])]
print(json.dumps([sorted(repr(x) for x in eval(src).run()) for src in json.loads(sys.argv[3])]))
"""


def test_lowered_joins_probes_and_sorts_agree_with_the_reference(monkeypatch):
    """Reduce-side joins (inner / left) over lowered inputs, the cross_set membership probe, sorts of whole
    records and of count frames, cross_right over a frame: this engine's lowered paths vs the reference."""
    import numpy as np
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    from dampr_b200.inputs import ArrayKVInput
    rng = random.Random(23)
    keys = [rng.randint(0, 60) for _ in range(3000)]
    vals = [rng.randint(-100, 100) for _ in range(3000)]
    k2 = [rng.randint(30, 90) for _ in range(500)]
    v2 = [rng.randint(0, 5) for _ in range(500)]
    A_ref="Dampr.memory(recs, partitions=3)"; B_ref="Dampr.memory(recs2, partitions=2)"
    A_our="Dampr.read_input(ArrayKVInput(K, V))"; B_our="Dampr.read_input(ArrayKVInput(K2, V2))"
    tmpl=[
     "{A}.group_by(lambda x: x[0], lambda x: x[1]).join({B}.group_by(lambda x: x[0], lambda x: x[1])).reduce(lambda l, r: (sum(l), sum(r)))",
     "{A}.group_by(lambda x: x[0], lambda x: x[1]).join({B}.group_by(lambda x: x[0], lambda x: x[1])).left_reduce(lambda l, r: (sum(l), sorted(r)))",
     "{A}.a_group_by(lambda x: x[0], lambda x: x[1]).sum().join({B}.count(lambda x: x[0])).reduce(lambda l, r: (list(l), list(r)))",
     "{A}.group_by(lambda x: x[0], lambda x: x[1]).reduce(lambda k, it: sum(it)).join({B}.group_by(lambda x: x[0], lambda x: x[1]).reduce(lambda k, it: max(it))).reduce(lambda l, r: next(l)[1] * next(r)[1])",
     "{B}.map(lambda x: x[0]).cross_set({A}, lambda b, table: (b[0], b[1], b[0] in table), agg=set)",
     "{B}.map(lambda x: x[0]).cross_set({A}, lambda b, table: b[0] not in table, agg=set)",
     "{A}.count(lambda x: x[0]).sort_by(lambda kc: -kc[1]).map(lambda kc: kc[0])",
     "{A}.sort_by(lambda x: x[1])",
     "{A}.sort_by(lambda x: -x[0])",
     "{A}.a_group_by(lambda x: x[0], lambda x: x[1]).sum().cross_right({B}.len(), lambda kv, n: (kv[0], kv[1] * n))",
    ]
    ref = reference("lowered_joins_probes_and_sorts", TWO_DRIVER, json.dumps(list(zip(keys, vals))),
                    json.dumps([t.format(A=A_ref, B=B_ref) for t in tmpl]), json.dumps(list(zip(k2, v2))))
    ns = {"Dampr": Dampr, "ArrayKVInput": ArrayKVInput, "K": np.array(keys, dtype=np.int64), "V": np.array(vals, dtype=np.int64),
          "K2": np.array(k2, dtype=np.int64), "V2": np.array(v2, dtype=np.int64)}
    seen = set()
    for t, exp in zip(tmpl, ref):
        monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
        monkeypatch.setattr(plan, "_BUFFERS", {})
        got = sorted(repr(x) for x in eval(t.format(A=A_our, B=B_our), ns).run())
        seen.update(h for _s, h, _d in runner_mod.LAST_STATS.stages)
        assert got == exp, t
    for needle in ("device join ranges", "device broadcast hash build+probe", "partition+sort of whole records",
                   "device sort of frame rows", "memoised per distinct"):
        assert any(needle in h for h in seen), needle


@pytest.mark.parametrize("path_kind", ["host-map", "scan-plumbing"])
def test_directory_inputs_agree_with_the_reference(path_kind, monkeypatch, tmp_path):
    """Dampr.text on a directory tree: several files laid out back to back, an empty file, files without a
    final newline, a .gz member."""
    import gzip
    import math
    import re
    import fake_device as F
    from oracle import gen
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    RX = re.compile(r"[^\w]+")
    d = tmp_path / "corpus"
    (d / "sub" / "deep").mkdir(parents=True)
    files = {"a.txt": gen.text(1, 150, V=80), "b.txt": gen.dirty_text(2, 120, 100), "sub/c.txt": b"tail without newline",
             "sub/deep/d.txt": b"", "sub/e.txt": gen.text(3, 60, V=40)[:-1]}
    for fn, data in files.items():
        (d / fn).write_bytes(data)
    with gzip.open(str(d / "sub" / "f.txt.gz"), "wb") as f:
        f.write(gen.text(4, 80, V=50))
    longest = max(len(l) + 1 for data in files.values() for l in data.split(b"\n")) + 5
    srcs = text_pipelines(900, 12, longest)
    ref = reference("directory_inputs", TEXT_DRIVER, str(d), json.dumps(srcs))
    monkeypatch.setattr(plan, "_pinned_ring", lambda n, b: [F.FakePinned(b) for _ in range(n)])
    for src, exp in zip(srcs, ref):
        monkeypatch.setattr(runner_mod, "_CTX", {settings.device: F.FakeCtx() if path_kind == "host-map" else F.FakeTextCtx()})
        monkeypatch.setattr(plan, "_BUFFERS", {})
        got = sorted(repr(x) for x in eval(src, {"Dampr": Dampr, "path": str(d), "RX": RX, "math": math}).run())
        assert got == exp, src


@pytest.mark.parametrize("path_kind", ["host-map", "scan-plumbing"])
def test_crlf_gzip_inputs_agree_with_the_reference(path_kind, monkeypatch, tmp_path):
    """.gz text is read in BINARY mode by the reference (dataset.py:488-493): only '\\n' ends a line, the '\\r'
    of a CRLF file stays in the line (so the tf-idf tokeniser yields a '' token per line and 'hello world\\r'
    is the line), a lone '\\r' does not end a line. Both as a gz-only directory (stays lowered: the CR flag is
    data there) and next to a plain CRLF file (universal newlines apply to that one)."""
    import gzip
    import math
    import re
    import fake_device as F
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    RX = re.compile(r"[^\w]+")
    crlf = b"hello world\r\nfoo bar\r\nlone\rcr inside\r\n\r\nlast line no cr\nunterminated\r"
    for layout in ("gz-only", "mixed"):
        d = tmp_path / layout
        d.mkdir()
        with gzip.open(str(d / "a.txt.gz"), "wb") as f:
            f.write(crlf)
        with gzip.open(str(d / "b.txt.gz"), "wb") as f:
            f.write(b"plain gz\nno carriage returns\n")
        if layout == "mixed":
            (d / "c.txt").write_bytes(b"text mode\r\nuniversal newlines\rhere\n")
        srcs = ["Dampr.text(path, 1 << 20)" + tail for tail in (
            ".flat_map(lambda x: x.split()).count()",
            ".flat_map(lambda x: set(RX.split(x.lower()))).count()",
            ".flat_map(lambda x: RX.split(x.lower())).count()",
            ".len()",
            ".map(lambda x: x)",
        )]
        ref = reference("crlf_gzip_" + layout, TEXT_DRIVER, str(d), json.dumps(srcs))
        assert repr("hello world\r") in ref[4] if layout == "gz-only" else True
        monkeypatch.setattr(plan, "_pinned_ring", lambda n, b: [F.FakePinned(b) for _ in range(n)])
        for src, exp in zip(srcs, ref):
            monkeypatch.setattr(runner_mod, "_CTX", {settings.device: F.FakeCtx() if path_kind == "host-map" else F.FakeTextCtx()})
            monkeypatch.setattr(plan, "_BUFFERS", {})
            got = sorted(repr(x) for x in eval(src, {"Dampr": Dampr, "path": str(d), "RX": RX, "math": math}).run())
            assert got == exp, (layout, src)
            if path_kind == "scan-plumbing" and layout == "gz-only" and "count" in src:
                assert any("device text tokenise+combine" in h for _s, h, _d in runner_mod.LAST_STATS.stages), src


def test_lowered_join_idioms_agree_with_the_reference(monkeypatch):
    """Columnar reduce-side joins (plan._lower_join): per-side folds (inner and left), and itertools.product over a
    right side with unique keys (many=True) — vs the reference's InnerJoin / LeftJoin (base.py:264-315). Joins whose
    aggregate is not an idiom, or whose right side has duplicate keys under product, take the generic path and
    must agree as well."""
    import itertools
    import numpy as np
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    from dampr_b200.inputs import ArrayKVInput
    rng = random.Random(41)
    keys = [rng.randint(0, 400) for _ in range(5000)]
    vals = [rng.randint(-100, 100) for _ in range(5000)]
    k2 = rng.sample(range(200, 700), 300)          # unique keys, about half of them present on the left
    v2 = [rng.randint(0, 50) for _ in range(300)]
    A_ref = "Dampr.memory(recs, partitions=3)"; B_ref = "Dampr.memory(recs2, partitions=2)"
    A_our = "Dampr.read_input(ArrayKVInput(K, V))"; B_our = "Dampr.read_input(ArrayKVInput(K2, V2))"
    G = ".group_by(lambda x: x[0], lambda x: x[1])"
    tmpl = [
        "{A}" + G + ".join({B}" + G + ").reduce(lambda l, r: (sum(l), len(list(r))))",
        "{A}" + G + ".join({B}" + G + ").reduce(lambda l, r: (max(l), min(r)))",
        "{A}" + G + ".join({B}" + G + ").reduce(lambda l, r: (len(list(l)), sum(r)))",
        "{A}" + G + ".join({B}" + G + ").left_reduce(lambda l, r: (sum(l), len(list(r))))",
        "{A}" + G + ".join({B}" + G + ").left_reduce(lambda l, r: (min(l), sum(r)))",
        "{A}" + G + ".join({B}" + G + ").reduce(lambda l, r: itertools.product(l, r), many=True)",
        "{B}" + G + ".join({A}" + G + ").reduce(lambda l, r: itertools.product(l, r), many=True)",   # duplicate right keys
        "{A}" + G + ".join({B}" + G + ").reduce(lambda l, r: (sum(l), sorted(r)))",                   # not an idiom
    ]
    driver = TWO_DRIVER.replace("import sys, json", "import sys, json, itertools")
    ref = reference("lowered_join_idioms", driver, json.dumps(list(zip(keys, vals))),
                    json.dumps([t.format(A=A_ref, B=B_ref) for t in tmpl]), json.dumps(list(zip(k2, v2))))
    ns = {"Dampr": Dampr, "ArrayKVInput": ArrayKVInput, "itertools": itertools, "K": np.array(keys, dtype=np.int64),
          "V": np.array(vals, dtype=np.int64), "K2": np.array(k2, dtype=np.int64), "V2": np.array(v2, dtype=np.int64)}
    hows = []
    for t, exp in zip(tmpl, ref):
        monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
        monkeypatch.setattr(plan, "_BUFFERS", {})
        got = sorted(repr(x) for x in eval(t.format(A=A_our, B=B_our), ns).run())
        hows.append([h for _s, h, _d in runner_mod.LAST_STATS.stages])
        assert got == exp, t
    for i in range(5):
        assert any("device join: per-side partition+sort+fold" in h for h in hows[i]), tmpl[i]
    assert any("device join: broadcast hash build + probe" in h for h in hows[5])
    for i in (6, 7):
        assert not any("device join:" in h for h in hows[i]), tmpl[i]


def test_lowered_topk_unique_prefix_agree_with_the_reference(monkeypatch):
    """The lowerings added for SURVEY §8(f)2 — topk over a frame (plan._lower_topk), group_by(...).unique() over kv
    records (plan._lower_unique), prefix / suffix / map_keys through the frame map — against the reference's own
    topk (dampr.py:621-652), unique (:727-746) and prefix / suffix (:310-340) on the same records. unique()'s value
    order inside a group is the reference's merge order, which depends on its worker scheduling: one input
    partition keeps it the input order, which is what the lowering produces."""
    import numpy as np
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    from dampr_b200.inputs import ArrayKVInput
    rng = random.Random(77)
    keys = [rng.randint(0, 300) for _ in range(6000)]
    vals = [rng.randint(-40, 40) for _ in range(6000)]
    A_ref = "Dampr.memory(recs, partitions=1)"
    A_our = "Dampr.read_input(ArrayKVInput(K, V))"
    G = ".group_by(lambda x: x[0], lambda x: x[1])"
    S = ".a_group_by(lambda x: x[0], lambda x: x[1]).sum()"
    tmpl = [
        "{A}" + S + ".topk(7, lambda x: x[1])",
        "{A}" + S + ".topk(40, lambda x: -x[1])",
        "{A}" + S + ".topk(1000, lambda x: x[0])",          # k larger than the frame
        "{A}" + S + ".topk(5, lambda x: x[1] * 2 - x[0])",  # not a projection: host heap
        "{A}" + S + ".map(lambda x: x[1]).topk(9)",                                   # a map fused in front of the topk
        "{A}" + S + ".filter(lambda x: x[0] % 2 == 0).map(lambda x: (x[1], x[0])).topk(6, lambda x: -x[0])",
        "{A}" + G + ".unique()",
        "{A}" + G + ".unique(lambda v: v % 3)",              # numeric key function: evaluated column-at-a-time
        "{A}" + G + ".unique(lambda v: str(v)[-1])",          # not numeric: host reducer over device-grouped records
        "{A}" + S + ".prefix(lambda x: x[1] % 10)",
        "{A}" + S + ".suffix(lambda x: x[0] + x[1])",
        "{A}" + S + ".map_keys(lambda k: k * 2).map_values(lambda v: v - 1)",
        "{A}" + S + ".map(lambda x: (x[0], x[1], x[1] / 7.0)).sink_json(__import__('tempfile').mkdtemp())",
        "{A}" + S + ".map(lambda x: x[1] * 0.5).sink_json(__import__('tempfile').mkdtemp())",
    ]
    ref = reference("lowered_topk_unique_prefix", TWO_DRIVER, json.dumps(list(zip(keys, vals))),
                    json.dumps([t.format(A=A_ref) for t in tmpl]), json.dumps([]))
    ns = {"Dampr": Dampr, "ArrayKVInput": ArrayKVInput, "K": np.array(keys, dtype=np.int64), "V": np.array(vals, dtype=np.int64)}
    hows = []
    for t, exp in zip(tmpl, ref):
        monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
        monkeypatch.setattr(plan, "_BUFFERS", {})
        got = sorted(repr(x) for x in eval(t.format(A=A_our), ns).run())
        hows.append([h for _s, h, _d in runner_mod.LAST_STATS.stages])
        assert got == exp, t
    for i in (0, 1, 2):
        assert any("device top-k candidates" in h for h in hows[i]), tmpl[i]
    assert not any("device top-k" in h for h in hows[3])
    for i in (4, 5):
        assert any("device top-k candidates" in h for h in hows[i]), (tmpl[i], hows[i])
    assert any("device unique" in h for h in hows[6]) and any("device unique" in h for h in hows[7])
    assert not any("device unique" in h for h in hows[8])
    for i in (9, 10, 11):
        assert any("frame map/filter evaluated column-at-a-time" in h for h in hows[i]), (tmpl[i], hows[i])
    for i in (12, 13):
        assert any("native frame sink" in h for h in hows[i]), (tmpl[i], hows[i])


def test_chains_over_binary_kv_inputs_agree_with_the_reference(monkeypatch):
    """Stages over binary (key, value) inputs that are more than a bare keyed fold — a map / filter chain in front of
    it, mean(), topk, a plain map, len() — run column-at-a-time on the two input columns (plan._lower_map: the kv
    input as a frame of (key, value) rows). Same records through the reference as Dampr.memory tuples."""
    import numpy as np
    from fake_device import FakeCtx
    from dampr_b200 import Dampr, settings, plan
    from dampr_b200 import runner as runner_mod
    from dampr_b200.inputs import ArrayKVInput
    rng = random.Random(99)
    keys = [rng.randint(0, 200) for _ in range(5000)]
    vals = [rng.randint(-30, 60) for _ in range(5000)]
    A_ref = "Dampr.memory(recs, partitions=3)"
    A_our = "Dampr.read_input(ArrayKVInput(K, V))"
    tmpl = [
        "{A}.len()",
        "{A}.mean(lambda x: x[0], lambda x: x[1])",
        "{A}.filter(lambda x: x[1] > 0).count(lambda x: x[0])",
        "{A}.map(lambda x: (x[0] % 10, x[1] * 2)).a_group_by(lambda x: x[0], lambda x: x[1]).sum()",
        "{A}.filter(lambda x: x[0] % 3 == 1).map(lambda x: (x[0], x[1] - 1)).fold_by(lambda x: x[0], max, lambda x: x[1])",
        "{A}.topk(6, lambda x: x[1])",
        "{A}.topk(4, lambda x: -x[0])",
        "{A}.map(lambda x: x[0] * 1000 + x[1])",
        "{A}.filter(lambda x: x[1] == 7).map(lambda x: x[0])",
        "{A}.map(lambda x: (x[1], x[0])).sort_by(lambda x: x[0])",
        "{A}.a_group_by(lambda x: x[0] % 5, lambda x: x[1]).reduce(min)",
        "{A}.map(lambda x: x[1] / 4.0).a_group_by(lambda x: 1).reduce(max)",
    ]
    ref = reference("chains_over_binary_kv_inputs", TWO_DRIVER, json.dumps(list(zip(keys, vals))),
                    json.dumps([t.format(A=A_ref) for t in tmpl]), json.dumps([]))
    ns = {"Dampr": Dampr, "ArrayKVInput": ArrayKVInput, "K": np.array(keys, dtype=np.int64), "V": np.array(vals, dtype=np.int64)}
    hows = []
    for t, exp in zip(tmpl, ref):
        monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
        monkeypatch.setattr(plan, "_BUFFERS", {})
        got = sorted(repr(x) for x in eval(t.format(A=A_our), ns).run())
        hows.append([h for _s, h, _d in runner_mod.LAST_STATS.stages])
        assert got == exp, t
    assert any("record count of a columnar input" in h for h in hows[0])
    for i in range(1, 10):
        assert not any(h.startswith("host-map") for h in hows[i][:1]), (tmpl[i], hows[i])
    # the synthetic kv inputs of the benchmarks have keys all over the unsigned 64-bit range (gen.kv): such keys
    # may be projected and grouped on (bit equality), not computed with
    big = [(k * 0x9E3779B97F4A7C15) % (1 << 64) for k in keys[:2000]]   # (argv carries the records: keep it short)
    vals = vals[:2000]
    tmpl2 = [
        "{A}.mean(lambda x: x[0], lambda x: x[1])",
        "{A}.filter(lambda x: x[1] > 0).count(lambda x: x[0])",
        "{A}.map(lambda x: (x[0], x[1] * 3)).a_group_by(lambda x: x[0], lambda x: x[1]).sum()",
        "{A}.map(lambda x: x[0] % 7).count()",                      # arithmetic on such keys: host map
    ]
    ref2 = reference("chains_over_binary_kv_inputs_u64_keys", TWO_DRIVER, json.dumps(list(zip(big, vals))),
                     json.dumps([t.format(A=A_ref) for t in tmpl2]), json.dumps([]))
    ns["K"], ns["V"] = np.array(big, dtype=np.uint64), np.array(vals, dtype=np.int64)
    for i, (t, exp) in enumerate(zip(tmpl2, ref2)):
        monkeypatch.setattr(runner_mod, "_CTX", {settings.device: FakeCtx()})
        monkeypatch.setattr(plan, "_BUFFERS", {})
        got = sorted(repr(x) for x in eval(t.format(A=A_our), ns).run())
        assert got == exp, t
        first = [h for _s, h, _d in runner_mod.LAST_STATS.stages][0]
        assert first.startswith("host-map") == (i == 3), (t, first)
