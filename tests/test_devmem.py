"""Who owns CUDA resources (arap_flow_b200/csrc/devmem.cuh, DESIGN.md 4.7).  CPU only.

Only devmem.cuh allocates or frees memory, or creates or destroys a stream, an event or a graph.  Only the C ABI
functions that free a handle contain a delete expression.  Every carve the library makes with Layout
(tests/devmem_host.cpp, built with g++ against the header's CUDA-free part) puts each block at the offset the
hand-chained 256-byte arithmetic it replaced gave it, and keeps each block's byte count."""
import ctypes as C
import os
import re
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

CSRC = os.path.join(ROOT, "arap_flow_b200", "csrc")
SOURCES = (".cu", ".cuh", ".cpp", ".h")

# the owners: DevBuf, GrowBuf, the stream / event / graph handles and the workspace's stream
OWNERS = {"devmem.cuh"}
ALLOC = re.compile(r"\bcuda(?:(?:Malloc|Free)(?:Host)?|StreamCreate\w*|StreamDestroy|EventCreate\w*|EventDestroy"
                   r"|GraphInstantiate\w*|GraphDestroy|GraphExecDestroy)\s*\(")
# the functions that free a C ABI handle: the only places a delete expression may stand
C_ABI_FREES = {"arapb200_api.cu": {"arapb200_batch_create", "arapb200_batch_destroy"},
               "opt_api.cu": {"Opt_ProblemDelete", "Opt_PlanFree"}}
# a definition starting in column 0: its name is the last identifier before the first parenthesis
DEFINITION = re.compile(r"^[A-Za-z_][\w\s*&:<>,]*?\b(\w+)\s*\(", re.M)

C1 = 854 * 480  # C1 and C2 frames
SIZES = (6, 1021 * 7, C1)


def al(b):
    return (b + 255) & ~255


def test_only_the_owners_allocate():
    found = set()
    for top in ("arap_flow_b200", "include"):
        for d, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if not f.endswith(SOURCES):
                    continue
                with open(os.path.join(d, f), encoding="utf-8") as fh:
                    if ALLOC.search(fh.read()):
                        found.add(f)
    assert "devmem.cuh" in found
    assert found <= OWNERS, sorted(found - OWNERS)


def _code(text):
    """text with comments and string literals blanked (line numbers kept)"""
    return re.sub(r'//[^\n]*|/\*.*?\*/|"(?:\\.|[^"\\\n])*"', lambda m: re.sub(r"[^\n]", " ", m.group()), text,
                  flags=re.S)


def test_only_the_c_abi_frees_delete():
    stray, frees = [], set()
    for d, _, files in os.walk(CSRC):
        for f in files:
            if not f.endswith(SOURCES):
                continue
            with open(os.path.join(d, f), encoding="utf-8") as fh:
                code = _code(fh.read())
            defs = [(m.start(), m.group(1)) for m in DEFINITION.finditer(code)]
            for m in re.finditer(r"\bdelete\b", code):
                if code[:m.start()].rstrip().endswith("="):  # a deleted function
                    continue
                fn = max(((at, name) for at, name in defs if at < m.start()), default=(0, None))[1]
                if fn in C_ABI_FREES.get(f, ()):
                    frees.add(fn)
                else:
                    stray.append(f"{f}:{code.count(chr(10), 0, m.start()) + 1} in {fn}")
    assert not stray, stray
    assert frees == set().union(*C_ABI_FREES.values())  # the scan sees the deletes that are allowed


@pytest.fixture(scope="module")
def dm(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("dm") / "libdm.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-shared", "-fPIC", "-o", so,
                           os.path.join(HERE, "devmem_host.cpp")])
    L = C.CDLL(so)
    z, i, out = C.c_size_t, C.c_int, C.POINTER(C.c_size_t)
    L.dm_extras.argtypes = [z, out]
    L.dm_frames.argtypes = [z, z, out]
    L.dm_scene.argtypes = [z, z, z, z, z, i, out]
    L.dm_warp.argtypes = [z, i, i, out]
    L.dm_flatten.argtypes = [z, i, i, i, i, out]
    L.dm_composite.argtypes = [z, z, i, i, i, out]
    return L


def _call(fn, n_out, *args):
    out = (C.c_size_t * n_out)()
    fn(*args, out)
    return list(out)


def _chain(blocks):
    """offsets of the blocks (None = not taken) and the end, as `o_next = o + al(bytes)` chains computed them"""
    offs, cur = [], 0
    for b in blocks:
        offs.append(None if b is None else cur)
        cur += 0 if b is None else al(b)
    return offs, cur


def _same(got, blocks):
    offs, end = _chain(blocks)
    for g, o in zip(got, offs):
        if o is not None:
            assert g == o
    assert got[len(blocks)] == end
    return end


def test_pipeline_slot_buffers_keep_their_blocks(dm):
    for N in SIZES:
        # backward flow and occlusion of maxW x maxH (two cudaMalloc of 8 N and N, and 9 N of pinned staging)
        end = _same(_call(dm.dm_extras, 3, N), [8 * N, N])
        assert 9 * N <= end < 9 * N + 512
        for K in (1, 4, 19):
            F = N * K  # positions, two z-buffers, then the frames' rgb, mask, flow, bflow, occ, flow0
            end = _same(_call(dm.dm_frames, 9, N, K), [8 * F, 8 * N, 3 * F, F, 8 * F, 8 * F, F, 8 * F])
            assert 37 * F + 8 * N <= end < 37 * F + 8 * N + 8 * 256


def test_scene_layout(dm):
    W, H, bgW, bgH = 854, 480, 942, 568  # C2 over a background with a 44-pixel margin
    N = W * H
    for K in (0, 19):
        for rgb0 in (False, True):
            got = _call(dm.dm_scene, 8, W, H, bgW, bgH, K, int(rgb0))
            F = N * (K + 1)
            # SceneLayout as it was: rgb0 = bg + al(3 bgW bgH), flow = rgb0 + (rgb0 ? al(3N) : 0), ...
            bg = 0
            r0 = bg + al(3 * bgW * bgH)
            fl = r0 + (al(3 * N) if rgb0 else 0)
            rgb = fl + al(8 * F)
            mask = rgb + al(3 * F)
            bf = mask + al(F)
            occ = bf + al(8 * F)
            assert got == [bg, r0, fl, rgb, mask, bf, occ, occ + al(F)]


def test_warp_workspace(dm):
    for N in SIZES:
        for ex, occ in ((False, False), (True, False), (True, True)):
            got = _call(dm.dm_warp, 11, N, int(ex), int(occ))
            # warp_common as it was: o_in = 0, o_pos = o_in + up256(8N), ..., total = o_occ + (occ ? up256(N) : 0)
            o_in = 0
            o_pos = o_in + al(8 * N)
            o_z = o_pos + al(8 * N)
            o_rgb = o_z + al(4 * N)
            o_orgb = o_rgb + al(3 * N)
            o_m = o_orgb + al(3 * N)
            o_om = o_m + al(N)
            o_bf = o_om + al(N)
            o_fl = o_bf + (al(8 * N) if ex else 0)
            o_occ = o_fl + (al(8 * N) if occ else 0)
            total = o_occ + (al(N) if occ else 0)
            assert got == [o_in, o_pos, o_z, o_rgb, o_orgb, o_m, o_om, o_bf, o_fl, o_occ, total]


@pytest.mark.parametrize("n_layers", [1, 32])
def test_flatten_workspace(dm, n_layers):
    for N in SIZES:
        for bg in (False, True):
            for out_bflow, out_occ in ((False, False), (True, False), (False, True), (True, True)):
                ex = out_bflow or out_occ
                got = _call(dm.dm_flatten, 5 * n_layers + 7, N, n_layers, int(bg), int(out_bflow), int(out_occ))
                # the take() chain as it was: per layer flow, rgb, mask (, bflow if ex)(, src if out_occ), the
                # background if given, then the outputs
                layer = [8 * N, 3 * N, N, 8 * N if ex else None, N if out_occ else None]
                tail = [3 * N if bg else None, 8 * N, 3 * N, N, 8 * N if out_bflow else None, N if out_occ else None]
                end = _same(got, layer * n_layers + tail)
                # what it reserved: (n + 1) x per_layer + al(3N), tight with a background and both extras or none
                per_layer = al(8 * N) + al(3 * N) + al(N) + (al(8 * N) + al(N) if ex else 0)
                need = (n_layers + 1) * per_layer + al(3 * N)
                assert end <= need
                if bg and out_bflow == out_occ:
                    assert end == need


@pytest.mark.parametrize("n_layers", [1, 32])
def test_composite_workspace(dm, n_layers):
    for N in SIZES:
        NB = N + 7 * 1021
        for ex, out_occ in ((False, False), (True, False), (True, True)):
            got = _call(dm.dm_composite, 5 * n_layers + 7, N, NB, n_layers, int(ex), int(out_occ))
            layer = [8 * N, 3 * N, N, N, 8 * N if ex else None]
            tail = [3 * NB, 8 * N, 3 * N, N, 8 * N if ex else None, N if out_occ else None]
            end = _same(got, layer * n_layers + tail)
            # what it reserved, summed separately
            per_layer = al(8 * N) + al(3 * N) + 2 * al(N) + (al(8 * N) if ex else 0)
            need = (n_layers * per_layer + al(3 * NB) + al(8 * N) + al(3 * N) + al(N) + (al(8 * N) if ex else 0) +
                    (al(N) if out_occ else 0))
            assert end == need
