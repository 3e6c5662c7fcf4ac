"""CPU: host-side logic -- ABI surface, state_dict contract, seeded weights, segment sharding, and the
world_size-2 exemplar broadcast over gloo.  No compute call into libdvc.so is made without a GPU."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    import dvc

    hdr = open(os.path.join(ROOT, "include", "dvc.h")).read()
    declared = set(re.findall(r"\b(dvc_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no prototypes parsed"
    lib = dvc.load_library()
    for sym in sorted(declared):
        assert hasattr(lib, sym), f"{sym} declared in include/dvc.h but not exported by libdvc.so"
    assert declared == set(dvc.EXPORTED)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    import dvc

    with pytest.raises(dvc.DvcError):
        dvc.Context(0)
    from models.ColorVidNet import ColorVidNet

    with pytest.raises(dvc.DvcError):
        ColorVidNet(7)(torch.zeros(1, 7, 16, 16))


def test_state_dict_contract():
    from models.ColorVidNet import ColorVidNet
    from models.NonlocalNet import VGG19_pytorch, WarpNet
    from oracle.weights import make_state_dict, net_shapes

    for name, m in (("warp", WarpNet(1)), ("color", ColorVidNet(7)), ("vgg", VGG19_pytorch())):
        sd, ref = m.state_dict(), net_shapes(name)
        assert list(sd.keys()) == list(ref.keys())
        assert all(tuple(sd[k].shape) == tuple(ref[k]) for k in ref)
        m.load_state_dict(make_state_dict(name))  # strict load of the reference-keyed dict
        m.eval()
        assert all(isinstance(p, torch.nn.Parameter) for p in m.parameters())
    assert sum(v.numel() for v in make_state_dict("vgg").values()) == 20024384
    assert sum(v.numel() for v in make_state_dict("warp").values()) == 6917131
    assert sum(v.numel() for v in make_state_dict("color").values()) == 32802370


def test_seeded_weights_are_reproducible():
    from oracle.weights import make_lab, make_state_dict

    a, b = make_state_dict("warp", 0), make_state_dict("warp", 0)
    assert all(torch.equal(a[k], b[k]) for k in a)
    c = make_state_dict("warp", 1)
    assert not torch.equal(a["theta.weight"], c["theta.weight"])
    assert torch.equal(make_lab(5, 1, 16, 16), make_lab(5, 1, 16, 16))


def test_segment_bounds_cover_clip_contiguously():
    from dvc.clip import segment_bounds

    for F_ in (0, 1, 7, 8, 64, 65):
        for world in (1, 2, 3, 8):
            prev = 0
            sizes = []
            for r in range(world):
                s, e = segment_bounds(F_, world, r)
                assert s == prev and e >= s
                prev = e
                sizes.append(e - s)
            assert prev == F_ and max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        segment_bounds(8, 2, 2)


def test_legal_shapes():
    from oracle.dvc_oracle import legal_shape

    assert legal_shape(480, 864) and legal_shape(216, 384) and legal_shape(40, 64)
    assert not legal_shape(480, 854) and not legal_shape(36, 64)


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
from dvc.clip import broadcast_exemplar, segment_bounds
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[3]}", rank=int(sys.argv[4]), world_size=2)
rank = dist.get_rank()
n = 96 * 260
pack = torch.arange(n, dtype=torch.float32) if rank == 0 else torch.zeros(n)
broadcast_exemplar(pack, src=0)
assert torch.equal(pack, torch.arange(n, dtype=torch.float32))
s, e = segment_bounds(9, 2, rank)
got = [None, None]
dist.all_gather_object(got, (s, e))
assert got == [(0, 5), (5, 9)], got
# query-row-sharded correlation (dvc/clip.py: RowShardedCorrelation): handle exchange, row partition and the peer
# pointer table, with a stand-in context that emulates "peer memory" through per-rank files (no GPU in this test)
from dvc.clip import RowShardedCorrelation
import numpy as np
class FakeCtx:
    device = "cpu"
    def __init__(self, rank, tmp): self.rank, self.tmp, self.routes = rank, tmp, None
    def peer_buffer_create(self, nbytes):
        path = os.path.join(self.tmp, f"buf{self.rank}.bin"); np.zeros(nbytes // 4, np.float32).tofile(path)
        return 1000 + self.rank, path.encode().ljust(64, b"\0")
    def peer_buffer_open(self, handle): return 1000 + int(handle.rstrip(b"\0").decode()[-5])
    def peer_buffer_close(self, ptr): pass
    def debug_flag(self, name, value): pass
    def peer_buffer_destroy(self, ptr): pass
    def corr_set_peer_outputs(self, y4=(), sim=(), row0=0): self.routes = (list(y4), list(sim), row0) if y4 else self.routes
    def corr_softmax_warp(self, th, ph, V, T):
        y4, sim, row0 = self.routes
        for base in y4:  # "store into every rank's buffer": row r of the shard -> global row row0 + r
            path = os.path.join(self.tmp, f"buf{base - 1000}.bin")
            mm = np.memmap(path, np.float32, "r+")
            n = th.shape[2]
            mm[(row0) * 4:(row0 + n) * 4] = np.repeat(np.arange(row0, row0 + n, dtype=np.float32), 4)
            mm.flush()
    def raw_view(self, ptr, numel): return torch.from_numpy(np.fromfile(os.path.join(self.tmp, f"buf{ptr - 1000}.bin"), np.float32)[:numel].copy())
torch.cuda.synchronize = lambda *a, **k: None
N = 11
fc = FakeCtx(rank, sys.argv[5])
sh = RowShardedCorrelation(fc, N)
assert (sh.row0, sh.row1) == ((0, 6) if rank == 0 else (6, 11))
assert sh._y4 == [1000, 1001] and sh._sim == [1000 + N * 16, 1001 + N * 16]
y, sim = sh(torch.zeros(1, 256, N), torch.zeros(1, 256, 4), torch.zeros(1, 4, 3), 1e-10)
assert torch.equal(y[0, :, 0], torch.arange(N, dtype=torch.float32)), y[0, :, 0]   # both shards landed in MY buffer
sh.close()
dist.barrier(); dist.destroy_process_group()
print("OK", rank)
"""


def test_exemplar_broadcast_world2_gloo(tmp_path):
    """N>1 plumbing on CPU: rank 0's operand pack reaches rank 1 unchanged; segments tile the clip."""
    script = tmp_path / "w.py"
    script.write_text(_WORKER)
    pkg = os.path.join(ROOT, "deep-exemplar-based-video-colorization_b200")
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, pkg, port, str(r), str(tmp_path)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0 and "OK" in o, o


def test_dropin_import_resolution_with_reference_tree(tmp_path):
    """INTEGRATION.md §1: with the package ahead of the reference on sys.path, `models.NonlocalNet` /
    `models.ColorVidNet` are the drop-ins while `models.FrameColor` is still the reference's own file.  The reference tree
    is stood in for by its layout: `models/` without __init__.py, holding its own NonlocalNet / ColorVidNet (which fail if
    they are ever imported) and FrameColor."""
    ref = tmp_path / "reference"
    (ref / "models").mkdir(parents=True)
    for mod in ("NonlocalNet", "ColorVidNet"):
        (ref / "models" / f"{mod}.py").write_text(f"raise ImportError('the reference {mod} shadowed the drop-in')\n")
    (ref / "models" / "FrameColor.py").write_text("def frame_colorization(*args, **kwargs):\n    raise NotImplementedError\n")
    code = r"""
import os, sys
sys.path.insert(0, sys.argv[2]); sys.path.insert(0, sys.argv[1])
import models
models.__path__.append(os.path.join(sys.argv[2], "models"))
from models.NonlocalNet import VGG19_pytorch, WarpNet
from models.ColorVidNet import ColorVidNet
from models.FrameColor import frame_colorization
import models.NonlocalNet as N, models.FrameColor as F
assert sys.argv[1] in N.__file__, N.__file__
assert F.__file__.startswith(sys.argv[2]), F.__file__
assert "dvc" in N.__dict__            # the drop-in imports the ctypes binding, the reference's file does not
print("RESOLVED")
"""
    pkg = os.path.join(ROOT, "deep-exemplar-based-video-colorization_b200")
    out = subprocess.run([sys.executable, "-c", code, pkg, str(ref)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "RESOLVED" in out.stdout, out.stdout + out.stderr


def test_header_is_plain_c(tmp_path):
    """include/dvc.h is the drop-in boundary: it must compile as C99 (extern "C" only under __cplusplus, no C++ types),
    and every prototype must take plain pointers / sizes."""
    src = tmp_path / "t.c"
    src.write_text('#include "dvc.h"\nint main(void) { return dvc_version() == 0; }\n')
    inc = os.path.join(ROOT, "include")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", inc, str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    hdr = open(os.path.join(inc, "dvc.h")).read()
    code = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)  # prototypes only, comments stripped
    assert "torch" not in code.lower() and "std::" not in code and "at::" not in code and "Tensor" not in code
