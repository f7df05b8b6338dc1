"""CPU tests of the cross-match's host side: assign() on hand-written matrices, the file listing and the report."""
import os

import numpy as np

from describealign_b200 import pairing


def _result(path1, min_len=100):
    path1 = np.asarray(path1, np.int64)
    errors = np.full(path1.shape, None, object)
    errors[path1 < 0] = "description 0: track shorter than 82 frames"
    min_len = np.full(path1.shape, min_len, np.int64)
    return pairing.CrossMatch(points=np.maximum(path1, 0) * 3, path1=path1, min_len=min_len,
                              candidates=np.maximum(path1, 0) * 5, passes=(path1 >= min_len) & (path1 >= 0),
                              errors=errors)


def test_identity_agrees_with_name_order():
    pick = pairing.assign(_result([[900, 10, 20], [30, 800, 5], [0, 40, 700]]))
    assert pick.pairs == [(0, 0), (1, 1), (2, 2)]
    assert pick.unmatched_videos == [] and pick.unmatched_descriptions == [] and pick.disagreements == []


def test_swapped_names_are_flagged():
    pick = pairing.assign(_result([[10, 900], [800, 20]]))
    assert pick.pairs == [(0, 1), (1, 0)]
    assert pick.disagreements == [(0, 1), (1, 0)]


def test_total_path_length_is_maximised_over_passing_cells_only():
    # greedy would take (0, 0) = 1000 and leave video 1 without a passing description; the optimum pairs both
    pick = pairing.assign(_result([[1000, 990], [950, 50]]))
    assert pick.pairs == [(0, 1), (1, 0)]
    # a cell below the minimum is never chosen, even where it is the only one left
    pick = pairing.assign(_result([[500, 90], [400, 99]]))
    assert pick.pairs == [(0, 0)] and pick.unmatched_videos == [1] and pick.unmatched_descriptions == [1]


def test_stranger_and_missing_episode():
    # description 1 belongs to no video; videos 1 and 2 are described by descriptions 2 and 3 (one shifted by the
    # stranger in name order)
    pick = pairing.assign(_result([[900, 0, 0, 0], [0, 30, 850, 0], [0, 20, 0, 870]]))
    assert pick.pairs == [(0, 0), (1, 2), (2, 3)]
    assert pick.unmatched_descriptions == [1] and pick.unmatched_videos == []
    assert pick.disagreements == [(1, 2), (2, 3)]


def test_error_cells_never_pass():
    pick = pairing.assign(_result([[-1, 700], [-1, -1]]))
    assert pick.pairs == [(0, 1)] and pick.unmatched_videos == [1] and pick.unmatched_descriptions == [0]
    assert pick.disagreements == [(0, 1), (1, None)]


def test_more_videos_than_descriptions():
    pick = pairing.assign(_result([[0], [900]]))
    assert pick.pairs == [(1, 0)] and pick.unmatched_videos == [0]
    assert pick.disagreements == [(0, None), (1, 0)]


def test_list_files(tmp_path):
    for n in ("Ep 10.mkv", "Ep 2.mkv", "Ep 1.mkv"):
        (tmp_path / n).write_bytes(b"")
    (tmp_path / "sub").mkdir()
    files, natural = pairing.list_files(str(tmp_path))
    names = [os.path.basename(f) for f in files]
    assert names == (["Ep 1.mkv", "Ep 2.mkv", "Ep 10.mkv"] if natural else ["Ep 1.mkv", "Ep 10.mkv", "Ep 2.mkv"])
    one = str(tmp_path / "Ep 2.mkv")
    assert pairing.list_files(one)[0] == [one]


def test_report_names_the_disagreement():
    res = _result([[10, 900], [800, -1]])
    text = pairing.format_report(["a.mkv", "b.mkv"], ["x.wav", "y.wav"], res, pairing.assign(res))
    assert "a.mkv  <->  y.wav" in text and "b.mkv  <->  x.wav" in text
    assert "the name order disagrees" in text and "error: description 0" in text
