"""The integer tables and parsers on the sampling path (bit-exact rows of SURVEY 8 a11).

Label tables: ps_vae/utils.py:82-136 (Common Voice gender / age buckets, VCTK gender; unknown -> -1).
Target parsing: ps_vae/inference.py:128-132.  Output indexing: ps_vae/inference.py:154-156.
Target mixes (``--target_mix``): the weights become integer thresholds on a uint32 Philox word, so a draw is platform-independent.
"""
from __future__ import annotations

import json
import math
from fractions import Fraction
from typing import List, Sequence, Tuple, Union

_CV_AGE = {"teens": 0, "twenties": 0, "thirties": 1, "fourties": 1, "fifties": 1, "sixties": 2, "seventies": 2, "eighties": 2, "nineties": 2}
_CV_GENDER = {"male": 0, "female": 1, "other": 2}
_VCTK_GENDER = {"M": 0, "F": 1}


def map_cv_age_to_label(age) -> int:
    return _CV_AGE.get(age, -1)


def map_cv_gender_to_label(gender) -> int:
    return _CV_GENDER.get(gender, -1)


def map_vctk_gender_to_label(gender) -> int:
    return _VCTK_GENDER.get(gender, -1)


def parse_classifier_target(text: str) -> Union[int, dict]:
    """``--classifier_target`` of the inference CLI: JSON (a dict of label -> class) first, else an int."""
    try:
        return json.loads(text)
    except json.JSONDecodeError:
        return int(text)


def parse_target_mix(text: str) -> List[Tuple[Union[int, dict], float]]:
    """``--target_mix`` of the inference CLI: a JSON list of ``[target, weight]`` pairs, each target an int or a dict of label -> class."""
    try:
        mix = json.loads(text)
    except json.JSONDecodeError as e:
        raise ValueError(f"--target_mix is not valid JSON: {e}") from None
    if not isinstance(mix, list) or not mix:
        raise ValueError("--target_mix must be a non-empty JSON list of [target, weight] pairs")
    out = []
    for item in mix:
        if not (isinstance(item, list) and len(item) == 2 and isinstance(item[0], (int, dict)) and not isinstance(item[0], bool)
                and isinstance(item[1], (int, float)) and not isinstance(item[1], bool)):
            raise ValueError(f"--target_mix entry {item!r} is not a [target, weight] pair (target: int or dict of label -> class)")
        out.append((item[0], float(item[1])))
    return out


def mix_thresholds(weights: Sequence[float], max_entries: int = 64) -> Tuple[List[int], List[int]]:
    """``(kept, thresholds)`` of a target mix: the indices of the entries with a non-zero weight and the ``len(kept) - 1`` uint32
    thresholds ``floor(2**32 * cumsum_k / total)``, computed in exact rational arithmetic.  A row whose uint32 word ``u`` is below
    ``thresholds[k]`` (and not below an earlier one) takes entry ``kept[k]``; a word above all of them takes the last kept entry, so entry k
    is drawn with probability ``(thresholds[k] - thresholds[k - 1]) / 2**32``, within 2**-32 of its weight's share."""
    fr = []
    for w in weights:
        if isinstance(w, bool) or not isinstance(w, (int, float)) and not hasattr(w, "__float__"):
            raise TypeError(f"mix weight {w!r} is not a number")
        if isinstance(w, int):
            f = Fraction(w)
        else:
            x = float(w)
            if not math.isfinite(x):
                raise ValueError(f"mix weight {x} is not finite")
            f = Fraction(x)
        if f < 0:
            raise ValueError(f"mix weight {w} is negative")
        fr.append(f)
    kept = [i for i, f in enumerate(fr) if f > 0]
    if not kept:
        raise ValueError("a target mix needs at least one positive weight")
    if len(kept) > max_entries:
        raise ValueError(f"a target mix has at most {max_entries} entries with a positive weight, got {len(kept)}")
    total = sum(fr[i] for i in kept)
    thr, cum = [], Fraction(0)
    for i in kept[:-1]:
        cum += fr[i]
        thr.append(math.floor(cum * 2 ** 32 / total))
    return kept, thr


def sample_filename(i: int) -> str:
    """Row ``i`` of a sampled batch is saved as ``sample_{i}.pt``."""
    return f"sample_{i}.pt"


def load_yaml_config(path: str) -> dict:
    """ps_vae/utils.py:69-80."""
    import yaml

    with open(path, "r") as f:
        return yaml.safe_load(f)
