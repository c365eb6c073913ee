"""The reference's scorer protocol (espnet2/legacy/nets/scorer_interface.py:85-188) on the espnet_b200 classes.

Replay: tests/golden/scorer_replay.npz (tests/golden/make_golden_scorer_replay.py) holds every call the REFERENCE's own BatchBeamSearch made
into its own TransformerDecoder and CTCPrefixScorer while decoding the tiny / small fixtures: batch_init_state, batch_score /
batch_score_partial with the prefixes, candidate ids and the states it threads through, select_state with its index arguments,
final_score.  TransformerDecoder.batch_score / select_state and CTCPrefixScorer.batch_init_state / batch_score_partial / select_state
receive the same call sequence and must return the scores the reference's scorers returned.
CPU: C-ABI entry points emulated (tests/emu_backend.py) -> host logic of the protocol; GPU (-m gpu): the CUDA kernels.
Registry path (-m gpu, needs the reference's own files under oracle/_ref): espnet_b200.integration.register + the reference's own
Speech2Text on device="cuda"."""
import json
import os
import sys

import numpy as np
import pytest
import torch

from golden_util import GOLDEN_DIR, decode_params, decode_results, load

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _reference():
    """Import the reference (oracle/_ref, or a fresh copy when /root/reference is mounted); skip if neither exists."""
    sys.path.insert(0, ROOT)
    from oracle import install_ref

    if not install_ref.available():
        try:
            install_ref.install(verbose=False)
        except Exception:
            pass
    if not install_ref.available():
        pytest.skip("oracle/_ref is absent (python oracle/install_ref.py needs /root/reference)")
    install_ref.activate()


def _replay(model, case, dn, device):
    """Drive our decoder / CTC scorer through the reference search's recorded calls; compare every score matrix they return."""
    from espnet_b200 import CTCPrefixScorer

    rec = np.load(os.path.join(GOLDEN_DIR, "scorer_replay.npz"))
    log = json.loads(str(rec[f"{case}:{dn}:log"]))
    x = torch.from_numpy(load(case)[0]["enc"]).to(device)
    scorers = dict(decoder=model.decoder, ctc=CTCPrefixScorer(model.ctc, model.eos))
    states = {}

    def t(key):
        return torch.from_numpy(rec[key]).to(device)

    def get(h):   # a recorded handle, a list of per-hypothesis handles, or None
        return [states[v] for v in h] if isinstance(h, list) else (None if h is None else states[h])

    def put(h, v):
        if isinstance(h, list):
            assert len(h) == len(v)
            states.update(zip(h, v))
        else:
            states[h] = v

    for n, c in enumerate(log):
        d, what = scorers[c["scorer"]], f"call {n}: {c['scorer']}.{c['op']}"
        if c["op"] == "init":
            put(c["out"], d.batch_init_state(x))
            continue
        if c["op"] == "select":
            s = get(c["state"])
            put(c["out"], d.select_state(s, c["i"]) if c["new_id"] is None else d.select_state(s, c["i"], c["new_id"]))
            continue
        if c["op"] == "final":
            assert d.final_score(get(c["state"])) == c["value"], what
            continue
        ys = t(c["ys"])
        if c["op"] == "score":
            scores, new = d.batch_score(ys, get(c["state"]), x.expand(ys.shape[0], *x.shape))
            new = list(new)
        else:
            scores, new = d.batch_score_partial(ys, None if c["ids"] is None else t(c["ids"]), get(c["state"]), x)
        np.testing.assert_allclose(scores.float().cpu().numpy(), rec[c["scores"]], rtol=2e-4, atol=2e-4, err_msg=what)
        put(c["out"], new)
    cw = decode_params(load(case)[0], dn)["ctc_weight"]
    used = {c["scorer"] for c in log if c["op"] in ("score", "partial")}
    assert used == {k for k, weight in (("decoder", 1.0 - cw), ("ctc", cw)) if weight}


@pytest.mark.parametrize("dn", ["joint", "att", "ctc", "joint_pen"])
def test_reference_beam_search_drives_our_scorers_host_logic(dn, monkeypatch):
    import argparse

    import emu_backend
    import espnet_b200
    from gpu_util import refbuild

    emu_backend.install_search(monkeypatch)
    z, cfg, w = load("tiny")
    model = espnet_b200.build_model(argparse.Namespace(**refbuild.model_yaml(cfg)))
    model.load_state_dict(w, strict=True)
    _replay(model.eval(), "tiny", dn, "cpu")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["tiny", "small"])
@pytest.mark.parametrize("dn", ["joint", "att", "ctc", "joint_pen"])
def test_reference_beam_search_drives_our_scorers_cuda(case, dn):
    from gpu_util import build_cuda_model

    z, cfg, w = load(case)
    model, _ = build_cuda_model(cfg, w)
    _replay(model, case, dn, "cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("dn", ["joint", "att"])
def test_reference_speech2text_with_registered_b200_classes(dn, tmp_path):
    """config.yaml names the b200_ classes -> the reference's ASRTask.build_model builds them, the reference's Speech2Text (device cuda)
    encodes through them and its BatchBeamSearch scores through TransformerDecoder.batch_score; result == the reference-only fixture."""
    import yaml

    from gpu_util import refbuild

    _reference()
    from espnet_b200 import integration

    integration.register()
    from espnet2.bin.asr_inference import Speech2Text

    z, cfg, w = load("tiny")
    y = refbuild.model_yaml(cfg)
    y.update(frontend="b200_default", normalize="b200_utterance_mvn", encoder="b200_conformer", decoder="b200_transformer")
    y["encoder_conf"].pop("use_flash_attn", None); y["decoder_conf"].pop("use_flash_attn", None)
    path = str(tmp_path / "config.yaml")
    with open(path, "w") as f:
        yaml.safe_dump(y, f)
    kw = decode_params(z, dn)
    s2t = Speech2Text(asr_train_config=path, asr_model_file=None, device="cuda", dtype="float32", nbest=10, **kw)
    missing = s2t.asr_model.load_state_dict(w, strict=False)
    assert not [k for k in missing.unexpected_keys], missing
    s2t.asr_model.eval()
    res = s2t(z["wave"])
    gold = decode_results(z, dn)
    assert len(res) == len(gold)
    for (_, _, _, h), (yseq, score, _) in zip(res, gold):
        assert h.yseq.tolist() == yseq
        assert abs(float(h.score) - score) <= 2e-4 * max(1.0, abs(score))
