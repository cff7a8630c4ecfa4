"""specimine over many files in one run (specimine.mine_files, smx_hw_best_grouped): every `.mined` file must be the one
a run on that file alone writes.  The CPU tier injects a host stand-in for the grouped call (argmin of the exact ratio
d / m over oracle distances), as test_specimine.py injects hw_distances; the GPU tier runs the grouped kernel and checks
it against smx_hw_distances and the oracle."""
import gzip
import json
import os
import shutil
from fractions import Fraction

import numpy as np
import pytest

import helpers as H
from specimux_b200 import _lib, specimine, synth


def _cases():
    with gzip.open(os.path.join(H.HERE, "golden_specimine", "cases.json.gz"), "rt") as fh:
        return json.load(fh)


_dist_cache = {}


def _oracle_distance(p, k, t):
    from oracle import aligner
    key = (p, k, t)
    if key not in _dist_cache:
        _dist_cache[key] = aligner.align(p, t, "HW", "distance", k, None)["editDistance"]
    return _dist_cache[key]


def _select(dists, lens):
    """The selection rule of smx_hw_best_grouped over one entry's (distance, pattern length) pairs, with exact
    rationals: smallest d / m among d != -1 and m > 0, ties to the first.  Returns (index, d) or (-1, -1)."""
    best = (-1, -1, None)
    for i, (d, m) in enumerate(zip(dists, lens)):
        if d == -1 or m == 0:
            continue
        r = Fraction(d, m)
        if best[2] is None or r < best[2]:
            best = (i, d, r)
    return best[0], best[1]


def _host_best_grouped(dist_of):
    def run(patterns, max_dist, texts, grp_pat_off, grp_txt_off, grp_txt_idx, device=0):
        n = len(grp_txt_idx)
        best_pat, best_dist = np.full(n, -1, dtype=np.int32), np.full(n, -1, dtype=np.int32)
        for g in range(len(grp_pat_off) - 1):
            pats = range(int(grp_pat_off[g]), int(grp_pat_off[g + 1]))
            for e in range(int(grp_txt_off[g]), int(grp_txt_off[g + 1])):
                t = texts[int(grp_txt_idx[e])]
                d = [dist_of(patterns[i], max_dist[i], t) if patterns[i] else 0 for i in pats]
                best_pat[e], best_dist[e] = _select(d, [len(patterns[i]) for i in pats])
        return best_pat, best_dist, 0.0
    return run


def _oracle_hw_distances(patterns, max_dist, texts, device=0):
    out = np.empty((len(patterns), len(texts)), dtype=np.int32)
    for i, (p, k) in enumerate(zip(patterns, max_dist)):
        for j, t in enumerate(texts):
            out[i, j] = _oracle_distance(p, k, t)
    return out


def _small_tree(root):
    return synth.specimine_tree(root, n_fwd=2, n_rev=3, n_full=4, n_partial=3, n_other=3, amplicon=160, seed=5)


def _read(path):
    with open(path) as fh:
        return fh.read()


def _single_runs(index, paths, flags):
    out = {}
    for p in paths:
        specimine.main(["--index", index, "--fastq", p] + flags)
        out[p] = _read(p + ".mined")
        os.remove(p + ".mined")
    return out


FLAG_SETS = [[], ["--partial-forward"], ["--partial-forward", "--no-partial-reverse"], ["--min-identity", "0.75"],
             ["--min-identity", "0.9", "--partial-forward"]]


@pytest.mark.parametrize("flags", FLAG_SETS, ids=lambda f: " ".join(f) or "default")
def test_multi_file_equals_single_runs_on_synthetic_tree(flags, tmp_path, monkeypatch):
    root = str(tmp_path)
    paths = _small_tree(root)
    index = os.path.join(root, "index.txt")
    monkeypatch.setattr(specimine, "hw_distances", _oracle_hw_distances)
    monkeypatch.setattr(specimine, "hw_best_grouped", _host_best_grouped(_oracle_distance))
    want = _single_runs(index, paths, flags)
    assert any(want.values()), "the tree should give hits"
    specimine.main(["--index", index, "--fastq"] + paths + flags)
    for p in paths:
        assert _read(p + ".mined") == want[p], p


def test_multi_file_splits_calls_by_budget(tmp_path, monkeypatch):
    """A budget smaller than one group: one call per group, same files."""
    root = str(tmp_path)
    paths = _small_tree(root)
    index = os.path.join(root, "index.txt")
    calls = []
    host = _host_best_grouped(_oracle_distance)

    def counted(*a, **kw):
        calls.append(len(a[4]) - 1)
        return host(*a, **kw)
    monkeypatch.setattr(specimine, "hw_distances", _oracle_hw_distances)
    want = _single_runs(index, paths, ["--partial-forward"])
    monkeypatch.setattr(specimine, "hw_best_grouped", counted)
    monkeypatch.setattr(specimine, "_GROUP_BUDGET", 1)
    specimine.main(["--index", index, "--fastq"] + paths + ["--partial-forward"])
    assert calls == [1] * (2 * len(paths))
    for p in paths:
        assert _read(p + ".mined") == want[p], p
    calls.clear()
    monkeypatch.setattr(specimine, "_GROUP_BUDGET", 64 << 20)
    specimine.main(["--index", index, "--fastq"] + paths + ["--partial-forward"])
    assert calls == [2 * len(paths)]


def _materialise_with_extra(case, root):
    """The golden case's tree plus a second specimen file: a copy of the target under another specimen id with the
    target's barcodes, so that its `.mined` file is the golden one too."""
    for rel, text in case["files"].items():
        p = os.path.join(root, rel)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        with open(p, "w") as fh:
            fh.write(text)
    target = os.path.join(root, case["target"])
    extra = target[:-len(".fastq")] + "_extra.fastq"
    shutil.copyfile(target, extra)
    spec = specimine.extract_specimen_id(target)
    index = os.path.join(root, "index.txt")
    lines = _read(index).splitlines()
    row = next(line for line in lines[1:] if line.split("\t")[0] == spec)
    with open(index, "a") as fh:
        fh.write(spec + "_extra\t" + row.split("\t", 1)[1] + "\n")
    return index, [target, extra]


@pytest.mark.parametrize("idx", range(5))
def test_goldens_through_multi_file_route(idx, tmp_path, monkeypatch):
    case = _cases()[idx]
    index, paths = _materialise_with_extra(case, str(tmp_path))
    monkeypatch.setattr(specimine, "hw_best_grouped", _host_best_grouped(_oracle_distance))
    specimine.main(["--index", index, "--fastq"] + paths + case["flags"])
    for p in paths:
        assert _read(p + ".mined") == case["mined"], p


def test_bad_files_are_skipped_and_exit_one(tmp_path, monkeypatch, caplog):
    root = str(tmp_path)
    paths = _small_tree(root)
    index = os.path.join(root, "index.txt")
    missing = os.path.join(root, "full", "ITS", "NOT-INDEXED.fastq")
    shutil.copyfile(paths[0], missing)
    outside = os.path.join(root, "elsewhere", paths[1].rsplit(os.sep, 1)[1])
    os.makedirs(os.path.dirname(outside))
    shutil.copyfile(paths[1], outside)
    empty = os.path.join(root, "full", "ITS", "EMPTY.fastq")
    open(empty, "w").close()
    with open(index, "a") as fh:
        fh.write("EMPTY\tITS\t" + "\t".join(_read(index).splitlines()[1].split("\t")[2:]) + "\n")
    monkeypatch.setattr(specimine, "hw_distances", _oracle_hw_distances)
    monkeypatch.setattr(specimine, "hw_best_grouped", _host_best_grouped(_oracle_distance))
    good = [paths[0], paths[2], empty]
    want = _single_runs(index, good, [])
    assert want[empty] == ""
    with pytest.raises(SystemExit) as ei:
        specimine.main(["--index", index, "--fastq", paths[0], missing, outside, paths[2], empty])
    assert ei.value.code == 1
    for p in good:
        assert _read(p + ".mined") == want[p], p
    assert not os.path.exists(missing + ".mined") and not os.path.exists(outside + ".mined")
    assert "Could not find specimen NOT-INDEXED in index file" in caplog.text
    assert "Could not find 'full' directory in path" in caplog.text


def test_selection_rule():
    # equal ratios go to the first pattern, an empty pattern never wins, -1 never wins
    assert _select([10, 20], [100, 200]) == (0, 10)
    assert _select([20, 10], [200, 100]) == (0, 20)
    assert _select([0, 3], [0, 100]) == (1, 3)
    assert _select([-1, 5, 4], [10, 100, 50]) == (1, 5)
    assert _select([-1, 0], [10, 0]) == (-1, -1)


def test_empty_text_is_never_mined(tmp_path, monkeypatch):
    root = str(tmp_path)
    paths = _small_tree(root)
    rev = sorted(os.listdir(os.path.join(root, "partial", "ITS", "ITS1F-ITS4")))
    with open(os.path.join(root, "partial", "ITS", "ITS1F-ITS4", [r for r in rev if "_rev_" in r][0]), "a") as fh:
        fh.write("@empty-read x\n\n+\n\n")
    monkeypatch.setattr(specimine, "hw_best_grouped", _host_best_grouped(_oracle_distance))
    specimine.main(["--index", os.path.join(root, "index.txt"), "--fastq"] + paths)
    assert all("empty-read" not in _read(p + ".mined") for p in paths)


def test_no_gpu_means_no_grouped_search():
    lib = _lib.load()
    if lib.smx_device_count() > 0:
        pytest.skip("box has a GPU")
    with pytest.raises(_lib.SmxError) as ei:
        specimine.hw_best_grouped(["ACGT"], [1], ["ACGTT"], np.array([0, 1]), np.array([0, 1]), np.array([0]))
    assert ei.value.code == _lib.SMX_ERR_NO_DEVICE


def test_argument_errors_need_no_gpu():
    with pytest.raises(_lib.SmxError) as ei:
        specimine.hw_best_grouped(["A" * 4097], [1], ["ACGT"], np.array([0, 1]), np.array([0, 1]), np.array([0]))
    assert ei.value.code == _lib.SMX_ERR_ARG
    with pytest.raises(_lib.SmxError) as ei:
        specimine.hw_best_grouped(["ACGT"], [1], ["ACGT"], np.array([0, 1]), np.array([0, 1]), np.array([3]))
    assert ei.value.code == _lib.SMX_ERR_ARG
    # nothing to search: no device needed, every entry -1
    bp, bd, _ = specimine.hw_best_grouped([""], [1], ["ACGT"], np.array([0, 1]), np.array([0, 1]), np.array([0]))
    assert bp.tolist() == [-1] and bd.tolist() == [-1]


# ---------------------------------------------------------------------------------------------------------------- GPU

def _rnd(rng, n):
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n)].tobytes().decode()


def _mutate(rng, s, rate):
    out = []
    for ch in s:
        u = rng.random()
        if u < rate / 3:
            out.append("ACGT"[rng.integers(0, 4)])
        elif u < 2 * rate / 3:
            out.append(ch + "ACGT"[rng.integers(0, 4)])
        elif u >= rate:
            out.append(ch)
    return "".join(out)


def _check_against_matrix(patterns, ks, texts, gp, gt, gi, oracle=False):
    got_p, got_d, ms = specimine.hw_best_grouped(patterns, ks, texts, np.array(gp), np.array(gt), np.array(gi))
    assert ms >= 0
    dist = specimine.hw_distances(patterns, ks, texts) if patterns and texts else None
    if oracle:
        want_dist = _oracle_hw_distances(patterns, ks, texts)
        assert (dist == want_dist).all()
    bad = []
    for g in range(len(gp) - 1):
        pats = list(range(gp[g], gp[g + 1]))
        for e in range(gt[g], gt[g + 1]):
            t = gi[e]
            want = _select([int(dist[i, t]) for i in pats], [len(patterns[i]) for i in pats])
            if (int(got_p[e]), int(got_d[e])) != want:
                bad.append((g, e, t, (int(got_p[e]), int(got_d[e])), want))
    assert not bad, bad[:10]


@pytest.mark.gpu
def test_grouped_equals_argmin_over_distances_all_classes():
    """One group per pattern length, 1 .. 128 words (every (SW, W) class the launcher picks) at word boundaries and
    between; shared texts with N / lower-case bytes, empty texts, k from 0 to unbounded."""
    rng = np.random.default_rng(7)
    patterns, ks, gp = [], [], [0]
    lens = sorted({n for w in range(1, 129) for n in (32 * w - 31, 32 * w) if n <= 4096} | {1, 2, 33, 700, 703, 4095})
    base = _rnd(rng, 4200)
    for n in lens:
        for _ in range(2):
            p = (_mutate(rng, base[:n], 0.03) + base[n:])[:n]          # exactly n bytes
            patterns.append(p)
            ks.append(int(rng.choice([0, 1, max(1, len(p) // 10), len(p) // 5, -1])))
        gp.append(len(patterns))
    texts = ["", "acgtn" + base[:300], _rnd(rng, 50)]
    texts += [_rnd(rng, int(rng.integers(0, 40))) + _mutate(rng, base[:int(n)], 0.05) + _rnd(rng, 20)
              for n in rng.integers(1, 4200, size=12)]
    texts[5] = texts[5][:7] + "N" + texts[5][8:]
    gt, gi = [0], []
    for g in range(len(gp) - 1):
        gi += [int(x) for x in rng.choice(len(texts), size=int(rng.integers(1, 8)), replace=False)]
        gt.append(len(gi))
    _check_against_matrix(patterns, ks, texts, gp, gt, gi)


@pytest.mark.gpu
def test_grouped_equals_oracle_with_ties_and_empties():
    rng = np.random.default_rng(11)
    a = _rnd(rng, 400)
    # equal ratios: m = 100 at d = 10 and m = 200 at d = 20 in the same text (crafted by substitutions)
    p100, p200 = a[:100], a[100:300]
    t_sub = list(a)
    for pos in list(range(3, 100, 10)) + list(range(105, 300, 10)):
        t_sub[pos] = "ACGT"[("ACGT".index(t_sub[pos]) + 1) % 4]
    t_tie = "".join(t_sub)
    patterns = [p100, p200, "", p200, p100, "AC", "acgtN" + a[:60]]
    ks = [-1, -1, 5, -1, -1, 0, 10]
    texts = [t_tie, "", a, _rnd(rng, 90), "ACGTACGT"]
    gp = [0, 2, 3, 5, 5, 7]            # group 3 has no patterns
    gt = [0, 3, 5, 8, 10, 10]          # group 4 has no texts
    gi = [0, 1, 2, 0, 4, 0, 3, 1, 2, 4]
    _check_against_matrix(patterns, ks, texts, gp, gt, gi, oracle=True)
    bp, bd, _ = specimine.hw_best_grouped(patterns, ks, texts, np.array(gp), np.array(gt), np.array(gi))
    assert (int(bp[0]), int(bd[0])) == (0, 10)      # tie: the first pattern
    assert (int(bp[5]), int(bd[5])) == (0, 20)      # group 2 lists them the other way round: p200 first
    assert int(bp[3]) == -1                          # group 1 holds only the empty pattern


@pytest.mark.gpu
def test_grouped_many_small_groups_one_call():
    rng = np.random.default_rng(13)
    amps = [_rnd(rng, int(rng.integers(20, 900))) for _ in range(40)]
    texts = [_mutate(rng, amps[i % 40], 0.07) for i in range(400)] + [""]
    patterns, ks, gp, gt, gi = [], [], [0], [0], []
    for g in range(300):
        a = amps[int(rng.integers(0, 40))]
        for _ in range(int(rng.integers(0, 6))):
            p = _mutate(rng, a, 0.07)
            patterns.append(p)
            ks.append(int(len(p) * 0.15) if rng.random() < 0.9 else -1)
        gp.append(len(patterns))
        gi += [int(x) for x in rng.integers(0, len(texts), size=int(rng.integers(0, 30)))]
        gt.append(len(gi))
    _check_against_matrix(patterns, ks, texts, gp, gt, gi)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", FLAG_SETS, ids=lambda f: " ".join(f) or "default")
def test_multi_file_gpu_equals_single_gpu_runs(flags, tmp_path):
    root = str(tmp_path)
    paths = synth.specimine_tree(root, n_fwd=3, n_rev=8, n_full=6, n_partial=4, n_other=8, amplicon=700, seed=9)
    index = os.path.join(root, "index.txt")
    want = _single_runs(index, paths, flags)
    assert any(want.values())
    specimine.main(["--index", index, "--fastq"] + paths + flags)
    for p in paths:
        assert _read(p + ".mined") == want[p], p


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(5))
def test_goldens_through_multi_file_route_on_gpu(idx, tmp_path):
    case = _cases()[idx]
    index, paths = _materialise_with_extra(case, str(tmp_path))
    specimine.main(["--index", index, "--fastq"] + paths + case["flags"])
    for p in paths:
        assert _read(p + ".mined") == case["mined"], p
