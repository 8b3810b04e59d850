"""ncu target: a few D_opt_FW_away iterations at 500 x 50000 (one launch of the persistent loop, fw_persist_ring_kernel)."""
import os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import accbpg_and_fw_b200 as acc      # noqa: E402
fd, h, L, x0 = acc.D_opt_design(500, 50000, randseed=1)
acc.D_opt_FW_away(fd._Hd, torch.tensor(x0, device="cuda"), 1e-12, 12, verbose=False)
print("ok")
