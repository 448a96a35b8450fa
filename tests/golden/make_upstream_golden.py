"""Regenerates tests/golden/upstream_torchaudio.npz: the outputs of torchaudio's Tacotron 2 sub-modules (_Postnet, _Encoder
convolutions, _Prenet) loaded with the canonical synthetic oracle weights, on the seeded inputs tests/test_oracle_upstream.py
builds.  The test compares the oracle with these stored outputs, so it runs without torchaudio.  Needs torchaudio; run from
the repo root: python tests/golden/make_upstream_golden.py
"""
import os
import sys

import numpy as np
import torch
import torchaudio
import torchaudio.models.tacotron2 as ta

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle import synthetic  # noqa: E402
from tests.test_oracle_upstream import encoder_convs_input, postnet_input, prenet_input  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    torch.set_num_threads(1)
    m = synthetic.make_model(stop_bias=-8.0)
    out = {"digest": np.array(synthetic.state_dict_digest(m.state_dict())), "torchaudio_version": np.array(torchaudio.__version__)}

    ref = ta._Postnet(80, 512, 5, 5).eval()
    for i, cb in enumerate(m.postnet.convs):
        ref.convolutions[i][0].load_state_dict(cb.conv.state_dict())
        ref.convolutions[i][1].load_state_dict(cb.bn.state_dict())
    with torch.no_grad():
        out["postnet"] = ref(postnet_input().transpose(1, 2)).transpose(1, 2).numpy()

    ref = ta._Encoder(512, 3, 5).eval()
    for i, cb in enumerate(m.enc_prenet.convs):
        ref.convolutions[i][0].load_state_dict(cb.conv.state_dict())
        ref.convolutions[i][1].load_state_dict(cb.bn.state_dict())
    want = encoder_convs_input()
    with torch.no_grad():
        for conv in ref.convolutions:                  # [TA]:407-408 (eval: dropout is identity)
            want = torch.relu(conv(want))
    out["encoder_convs"] = want.numpy()

    ref = ta._Prenet(80, [256, 256]).eval()
    with torch.no_grad():
        ref.layers[0].weight.copy_(m.dec_prenet.fc1.weight)
        ref.layers[1].weight.copy_(m.dec_prenet.fc2.weight)
        torch.manual_seed(0)
        out["prenet"] = ref(prenet_input()).numpy()

    np.savez_compressed(os.path.join(HERE, "upstream_torchaudio.npz"), **out)
    print("torchaudio", torchaudio.__version__, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
