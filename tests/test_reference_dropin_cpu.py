"""Drop-in check against the reference's OWN call chain, pinned by tests/golden/dropin.npz (oracle/make_golden_dropin.py
ran models.networks.define_G, base_model.load_network and base_model.save_network of the unmodified reference):
define_G's `RDN_arch.bin_stage4_lstm()` must build OUR module with the reference's class and state_dict schema, and the
reference's checkpoint load / save steps must round-trip through it."""
import os
from collections import OrderedDict

import numpy as np
import pytest
import torch


def load_network_clean(load_net):
    """The key handling of base_model.load_network (base_model.py:89-103), if / if-else as written there."""
    clean = OrderedDict()
    for k, v in load_net.items():
        if k.startswith("module."):
            clean[k[7:]] = v
        if k.startswith("InterpNet."):
            clean[k[10:]] = v
        else:
            clean[k] = v
    return clean


def test_define_g_and_checkpoint_roundtrip(tmp_path, golden_dir):
    from oracle import bin_oracle as O
    import bin_b200.rdn as ours
    g = np.load(os.path.join(golden_dir, "dropin.npz"))
    netG = ours.bin_stage4_lstm()                                   # networks.py:9-10 for which_model_G 'bin_stage4'
    assert type(netG).__name__ == str(g["netG_class"])
    assert isinstance(netG, ours.RDN_residual_interp_5_input_ConvLSTM_L)
    state = netG.state_dict()
    assert list(state.keys()) == list(g["state_keys"])
    assert ["x".join(map(str, v.shape)) for v in state.values()] == list(g["state_shapes"])
    # checkpoint round trip through load_network's key handling.  'InterpNet.' is the prefix it really strips; its
    # 'module.' branch also re-adds the prefixed key, so a 'module.'-prefixed file fails the strict load with the
    # reference's own network as well.
    sd = O.synth_state_dict(2)
    ckpt = tmp_path / "ck_G.pth"
    torch.save({("InterpNet." + k): v for k, v in sd.items()}, ckpt)
    clean = load_network_clean(torch.load(ckpt))
    assert list(clean.keys()) == list(g["load_interpnet_keys"])
    netG.load_state_dict(clean, strict=True)
    assert torch.equal(netG.model.model2_3.GFF[0].weight, sd["model.model2_1.GFF.0.weight"])
    clean_m = load_network_clean({("module." + k): v for k, v in sd.items()})
    assert list(clean_m.keys()) == list(g["load_module_keys"])
    assert bool(g["load_module_strict_fails"])
    with pytest.raises(RuntimeError):
        netG.load_state_dict(clean_m, strict=True)
    # save_network writes the same schema back (base_model.py:79-87): state_dict, every tensor moved to the CPU
    out = netG.state_dict()
    for k, v in out.items():
        out[k] = v.cpu()
    torch.save(out, tmp_path / "7_G.pth")
    back = torch.load(tmp_path / "7_G.pth")
    assert list(back.keys()) == list(g["saved_keys"])
    assert all(torch.equal(back[k], sd[k]) for k in back)
