"""Generate tests/golden/scorer_replay.npz from the UNMODIFIED reference (run where the reference is available).

    python tests/golden/make_golden_scorer_replay.py

The reference's own BatchBeamSearch (wired as espnet2/bin/asr_inference.py:168-176 does) decodes the stored encoder output of the
tiny / small fixtures with the reference's own TransformerDecoder and CTCPrefixScorer.  Every call the search makes into the scorer
protocol (scorer_interface.py:85-188) is recorded: the method, its prefixes / candidate ids, which earlier states it was handed, the
scores it returned and the index arguments of select_state.  States are opaque to the search, so they are recorded as handles.
tests/test_scorer_interface.py replays the same call sequence on the espnet_b200 scorers and compares the scores.
"""
import json
import logging
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import refbuild  # noqa: E402
import refshim  # noqa: E402
from golden_util import decode_params, decode_results, load  # noqa: E402

logging.disable(logging.WARNING)
CASES = ("tiny", "small")
DECODES = ("joint", "att", "ctc", "joint_pen")


class _Handle:
    def __init__(self, hid, val):
        self.hid, self.val = hid, val


def recorder(inner, name, log, arrays, prefix):
    """A scorer with inner's interface that forwards every protocol call to inner and appends it to log."""
    from espnet2.legacy.nets.scorer_interface import BatchPartialScorerInterface, BatchScorerInterface

    counter = [0]

    def arr(a):
        key = f"{prefix}:{len(arrays)}"
        arrays[key] = a.detach().cpu().numpy()
        return key

    def wrap(v):   # one state -> one handle, whatever the scorer keeps inside it
        counter[0] += 1
        return _Handle(f"{name}{counter[0]}", v)

    def unwrap(v):   # the search passes a handle, a list of per-hypothesis handles, or None
        return [h.val for h in v] if isinstance(v, list) else (None if v is None else v.val)

    def ids_of(v):
        return [h.hid for h in v] if isinstance(v, list) else (None if v is None else v.hid)

    class Rec(BatchPartialScorerInterface if isinstance(inner, BatchPartialScorerInterface) else BatchScorerInterface):
        def batch_init_state(self, x):
            out = wrap(inner.batch_init_state(x))
            log.append(dict(op="init", scorer=name, out=ids_of(out)))
            return out

        def batch_score(self, ys, states, xs):
            scores, new = inner.batch_score(ys, unwrap(states), xs)
            new = [wrap(st) for st in new]
            log.append(dict(op="score", scorer=name, ys=arr(ys), state=ids_of(states), scores=arr(scores), out=ids_of(new)))
            return scores, new

        def batch_score_partial(self, ys, ids, state, xs):
            scores, new = inner.batch_score_partial(ys, ids, unwrap(state), xs)
            new = wrap(new)
            log.append(dict(op="partial", scorer=name, ys=arr(ys), ids=None if ids is None else arr(ids), state=ids_of(state),
                            scores=arr(scores), out=ids_of(new)))
            return scores, new

        def select_state(self, state, i, new_id=None):
            out = wrap(inner.select_state(unwrap(state), i, new_id) if new_id is not None else inner.select_state(unwrap(state), i))
            log.append(dict(op="select", scorer=name, state=ids_of(state), i=int(i), new_id=None if new_id is None else int(new_id),
                            out=ids_of(out)))
            return out

        def final_score(self, state):
            s = float(inner.final_score(unwrap(state)))
            log.append(dict(op="final", scorer=name, state=ids_of(state), value=s))
            return s

    return Rec()


def record(case, dn, out):
    from espnet2.legacy.nets.batch_beam_search import BatchBeamSearch
    from espnet2.legacy.nets.scorers.ctc import CTCPrefixScorer
    from espnet2.legacy.nets.scorers.length_bonus import LengthBonus

    z, cfg, w = load(case)
    model = refbuild.build_reference(cfg, seed=0).asr_model
    model.load_state_dict(w, strict=True)
    model.eval()
    kw = decode_params(z, dn)
    cw, V = kw["ctc_weight"], model.vocab_size
    log, prefix = [], f"{case}:{dn}"
    scorers = dict(decoder=recorder(model.decoder, "decoder", log, out, prefix),
                   ctc=recorder(CTCPrefixScorer(ctc=model.ctc, eos=model.eos), "ctc", log, out, prefix), length_bonus=LengthBonus(V))
    weights = dict(decoder=1.0 - cw, ctc=cw, lm=1.0, ngram=0.9, length_bonus=kw["penalty"])
    bs = BatchBeamSearch(beam_size=kw["beam_size"], weights=weights, scorers=scorers, sos=model.sos, eos=model.eos, vocab_size=V,
                         token_list=model.token_list, pre_beam_score_key=None if cw == 1.0 else "full", normalize_length=kw["normalize_length"])
    with torch.no_grad():
        hyps = bs(x=torch.from_numpy(z["enc"]), maxlenratio=kw["maxlenratio"], minlenratio=kw["minlenratio"])
    gold = decode_results(z, dn)   # what the reference's Speech2Text returned for the same fixture
    assert [h.yseq.tolist() for h in hyps[:len(gold)]] == [g[0] for g in gold], (case, dn)
    out[f"{prefix}:log"] = np.array(json.dumps(log))
    print(case, dn, len(log), "calls")


if __name__ == "__main__":
    refshim.install()
    out = {}
    for case in CASES:
        for dn in DECODES:
            record(case, dn, out)
    path = os.path.join(HERE, "scorer_replay.npz")
    np.savez_compressed(path, **out)
    print("->", path, os.path.getsize(path) // 1024, "KiB")
