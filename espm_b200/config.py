"""Run-time switches of espm_b200 (module-level so that the estimator keeps the reference's signature).

distributed : "auto" | True | False
    Shard the image rows over the ranks of the default torch.distributed process group.  "auto" shards
    whenever a process group with more than one rank is initialised.
device_init : bool
    When neither W nor H is passed to ``fit_transform``, run the randomized SVD of scikit-learn's NNDSVD
    initialisation on the device (init_device.py) instead of on the host.  Unsharded fits with n < p only.
x_storage : "auto" | "dense" | "uint8" | "uint16"
    Storage of X on the device.  "auto" keeps count data (integers below 256 / 65536, fp32 arithmetic, nothing for
    remove_zeros_lines / normalize to patch) as uint8 / uint16 and streams 4x / 2x fewer bytes per pass; "dense" always
    stores the uploaded floating-point values (what BASELINE.json's fp32 / fp64 roofline figures are quoted on).
speculate_h : bool
    simplex_H: espm_h_finish applies the lock-step bisection count of the previous H update right after its trace and
    espm_h_apply only confirms it (and redoes the replay when the count changed).  Results are identical either way;
    the tests compare the two bit for bit.
"""
import os as _os

distributed = "auto"
speculate_h = _os.environ.get("ESPM_B200_SPECULATE_H", "1") != "0"
x_storage = "auto"
device_init = True
