"""Generate tests/golden/dropin.npz by EXECUTING THE UNMODIFIED REFERENCE (laomao0/BIN) call chain that builds,
loads and saves the generator network:

    python oracle/make_golden_dropin.py /path/to/BIN

Recorded (names and key lists only; no reference source is stored):
  netG_class                 class of what models.networks.define_G returns for which_model_G 'bin_stage4' (networks.py:5-14)
  state_keys / state_shapes  netG.state_dict() keys in order and their shapes ("32x96x3x3")
  load_interpnet_keys        keys BaseModel.load_network hands to load_state_dict for an 'InterpNet.'-prefixed checkpoint
  load_module_keys           the same for a 'module.'-prefixed checkpoint (base_model.py:89-103), and
  load_module_strict_fails   whether that strict load fails on the reference's own network
  saved_keys                 keys of the file BaseModel.save_network writes (base_model.py:79-87)
tests/test_reference_dropin_cpu.py checks bin_b200.rdn against them.
"""
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
if len(sys.argv) != 2 or not os.path.isfile(os.path.join(sys.argv[1], "models", "networks.py")):
    raise SystemExit(__doc__)
sys.path.insert(0, os.path.abspath(sys.argv[1]))

import models.networks as networks            # noqa: E402  (the reference itself)
from models.base_model import BaseModel       # noqa: E402
from oracle import bin_oracle as O            # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden", "dropin.npz")


def load_network_keys(net, ckpt_sd, path):
    """Run BaseModel.load_network on `ckpt_sd`, recording the dict it passes to load_state_dict."""
    seen = {}
    real = net.load_state_dict

    def record(sd, strict=True):
        seen["keys"] = list(sd.keys())
        return real(sd, strict=strict)
    torch.save(ckpt_sd, path)
    bm = BaseModel.__new__(BaseModel)
    bm.device = torch.device("cpu")
    net.load_state_dict = record
    try:
        BaseModel.load_network(bm, path, net, strict=True)
        failed = False
    except RuntimeError:
        failed = True
    finally:
        del net.load_state_dict
    return seen["keys"], failed


def main():
    opt = {"network_G": {"which_model_G": "bin_stage4", "nframes": 6, "version": 2}}
    net = networks.define_G(opt)
    sd = O.synth_state_dict(2)
    state = net.state_dict()
    with tempfile.TemporaryDirectory() as tmp:
        ki, fi = load_network_keys(net, {"InterpNet." + k: v for k, v in sd.items()}, os.path.join(tmp, "a.pth"))
        km, fm = load_network_keys(net, {"module." + k: v for k, v in sd.items()}, os.path.join(tmp, "b.pth"))
        assert not fi and fm
        bm = BaseModel.__new__(BaseModel)
        bm.opt = {"path": {"models": tmp}}
        BaseModel.save_network(bm, net, "G", 7)
        saved = list(torch.load(os.path.join(tmp, "7_G.pth")).keys())
    np.savez_compressed(OUT, netG_class=np.array(type(net).__name__),
                        state_keys=np.array(list(state.keys())),
                        state_shapes=np.array(["x".join(map(str, v.shape)) for v in state.values()]),
                        load_interpnet_keys=np.array(ki), load_module_keys=np.array(km),
                        load_module_strict_fails=np.array(fm), saved_keys=np.array(saved))
    print("wrote", OUT, os.path.getsize(OUT), "bytes:", type(net).__name__, len(state), "keys")


if __name__ == "__main__":
    main()
