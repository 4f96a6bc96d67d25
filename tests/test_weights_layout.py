"""percepnet_b200.weights.pack_state_dict against the reference's real exporter (dump_percepnet.py): the exporter's
own monkey-patched `dump_data` methods, run on the reference's PercepNet module carrying synth_state_dict(3), emitted
C arrays whose digests tests/golden/make_golden.py stored in tests/golden/reference_digests.json, with the module's
state_dict shapes and layer order.  Our packed arrays must equal the emitted ones exactly.  CPU."""
from util import digest, reference_digests


def test_pack_matches_reference_exporter():
    from percepnet_b200.weights import LAYERS, pack_state_dict, synth_state_dict
    gold = reference_digests()["exporter"]
    sd = synth_state_dict(3)
    assert {k: list(v.shape) for k, v in sd.items()} == gold["state_dict_shapes"]   # names of rnn_train.py:111-121
    packed = pack_state_dict(sd)
    # the big 512x512 GRUs share code with gru_rb: the cheap layers and one big GRU were dumped
    assert gold["arrays"]
    for key, want in gold["arrays"].items():
        assert digest(packed.arrays[key].ravel()) == want, key
    assert [l[0] for l in LAYERS] == gold["layers"]                                   # RNNModel field order
