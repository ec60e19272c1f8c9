"""CPU restatement of tracks from frame 0 (DESIGN.md 4.9), for the tests.

Built on tests/sequence_oracle.py (interp with the pixel grid as the vertex source, and the frame sequence itself),
tests/occlusion_oracle.py (the occlusion rule) and tests/background_oracle.py (the composite over a moving background);
the only new rules are the scene's owner selection of the flow and the query gather.  numpy float32, one rounding per
operation, so it can be compared with the CUDA kernels bit for bit.  Held to analytic cases by tests/test_oracle_tracks.py.
"""
import numpy as np

from oracle import pyoracle as O
from tests import background_oracle as BO
from tests import occlusion_oracle as OO
from tests import sequence_oracle as SO

F = np.float32
KEYS = ("flow0", "bflow0", "occ0")


def tracks(positions, seq, mask_red):
    """One problem's tracks from P_1 .. P_K = positions and their frame sequence `seq` (sequence_oracle.warp_seq's dict,
    which carries flow0 and the splat indices): flow0[k] = P_k - grid, bflow0[k] = interp(z_k, P_k, grid), occ0[k] = the occlusion rule with p's
    surface from the input mask and q's from z_k.  Returns a dict of [K, ...] arrays (KEYS)."""
    K, H, W = seq["splat"].shape
    g = O.grid(W, H)
    seg = np.where(np.asarray(mask_red) == 0, 0, -1)
    out = {k: [] for k in KEYS}
    for k in range(K):
        z = seq["splat"][k]
        bflow0 = SO.interp(z, np.asarray(positions[k], F), g)
        out["flow0"].append(seq["flow0"][k])
        out["bflow0"].append(bflow0)
        out["occ0"].append(OO.occlusion(seg, [seq["flow0"][k]], [bflow0], np.where(z != 0, 0, -1)))
    return {k: np.stack(v) for k, v in out.items()}


def warp_tracks(positions, mask_red):
    """What arapb200_warp_tracks computes (and the sequence it comes from).  Returns (tracks dict, seq dict)."""
    H, W = mask_red.shape
    seq = SO.warp_seq(positions, np.zeros((H, W, 3), np.uint8), mask_red)
    return tracks(positions, seq, mask_red), seq


def owner(src_masks, shape):
    """The last layer whose input mask has p on the object, -1 = the background."""
    own = np.full(shape, -1)
    for s, m in enumerate(src_masks):
        own[np.asarray(m) == 0] = s
    return own


def scene_tracks(layer_seqs, layer_tracks, src_masks, frame_motions):
    """A scene's tracks: per frame k, the composite (background_oracle.composite with the maps of motion_from = None,
    motion_to = A_k) of the layers' frame-k warped masks, flow0 and bflow0 over their input masks gives bflow0 and occ0;
    flow0 is the owner's flow0 on object pixels and A_k(p) - p elsewhere."""
    n = len(layer_seqs)
    K, H, W = layer_seqs[0]["mask"].shape
    own = owner(src_masks, (H, W))
    yy, xx = np.mgrid[0:H, 0:W]
    zeros = [np.zeros((H, W, 3), np.uint8)] * n
    out = {k: [] for k in KEYS}
    for k in range(K):
        flows = [t["flow0"][k] for t in layer_tracks]
        c = BO.composite(flows, zeros, [q["mask"][k] for q in layer_seqs], src_masks,
                         [t["bflow0"][k] for t in layer_tracks], np.zeros((1, 1, 3), np.uint8),
                         BO.coeffs(frame_motions[k]))
        mine = np.stack(flows)[np.maximum(own, 0), yy, xx]
        out["flow0"].append(np.where((own >= 0)[..., None], mine, c["flow"]).astype(F))   # c["flow"]: A_k(p) - p there
        out["bflow0"].append(c["bflow"])
        out["occ0"].append(c["occ"])
    return {k: np.stack(v) for k, v in out.items()}


def gather(tr, queries):
    """query_pos[k][i] = (x, y) + flow0[k][y, x] in float32, query_occ[k][i] = occ0[k][y, x]."""
    q = np.asarray(queries, np.int64).reshape(-1, 2)
    x, y = q[:, 0], q[:, 1]
    f = tr["flow0"][:, y, x]
    pos = np.stack([x.astype(F) + f[..., 0], y.astype(F) + f[..., 1]], -1)
    return dict(query_pos=pos.astype(F), query_occ=tr["occ0"][:, y, x])
