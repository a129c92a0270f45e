"""K5 wgrad kernel alone: random bf16 X / dY block-image stashes vs fp32 torch matmuls of the same operands
(exercises the MN-major operand reads, the 32-point slab pipeline, split-K atomics and the db column sums)."""
import pytest
import torch

from reflect_sampling_nerf_b200 import _lib, ops
from reflect_sampling_nerf_b200.blocks import pack_blocks, pack_blocks_cm

pytestmark = pytest.mark.gpu
STASH_BLOCKS, DY_BLOCKS = 41, 39
SWIZZLED_X_BLOCKS = (0, 1, 38)      # csrc/field_layout.cuh: STASH_ENC, STASH_IDE
# (dY first block, m_blocks, X first block, n_blocks, has_db) -- csrc/field_wgrad.cu kJobs
JOBS = [(7, 4, 0, 2, 1), (11, 4, 2, 4, 1), (15, 4, 6, 4, 1), (19, 4, 10, 4, 1), (23, 4, 0, 2, 0), (23, 4, 14, 4, 1),
        (27, 4, 18, 4, 1), (31, 4, 22, 4, 1), (35, 4, 26, 4, 1), None, (0, 3, 30, 4, 1), (0, 2, 39, 2, 0),
        None, (1, 2, 38, 1, 0)]
# jobs 9 (bottleneck x h7) and 12 (mid x bottleneck) are not computed by the kernel: rsn_field_wgrad_finish derives them
# from G = dY_mid^T h7 = rows 64-191 of job 10, which loads 3 dY blocks (seed, dY_mid) into an M = 256 accumulator (the
# last 64 rows are a by-product that nobody reads)


@pytest.mark.parametrize("n_tiles", [1, 3, 40])
def test_wgrad_matches_matmul(n_tiles):
    g = torch.Generator().manual_seed(n_tiles)
    pts = n_tiles * 128
    x = (torch.randn(pts, STASH_BLOCKS * 64, generator=g) * 0.5).bfloat16()
    dy = (torch.randn(pts, DY_BLOCKS * 64, generator=g) * 0.1).bfloat16()
    # stash layout: [tile][block][16 KB]; the encoding blocks (IPE 0-1, IDE 38) are swizzled images (pack_blocks gives
    # [K/64 blocks][rows][128] for a [rows, K] matrix), everything the epilogues write is chunk-major (pack_blocks_cm gives
    # [tile][K/64 blocks][16 KB]); each forward-stash tile is followed by 36,864 bytes of ReLU bit masks the wgrad does not read
    x_sw = torch.stack([pack_blocks(x[t * 128:(t + 1) * 128]).reshape(STASH_BLOCKS, 16384) for t in range(n_tiles)])
    x_img = pack_blocks_cm(x)
    for b in SWIZZLED_X_BLOCKS:
        x_img[:, b] = x_sw[:, b]
    xs = torch.cat([x_img.reshape(n_tiles, -1), torch.zeros(n_tiles, 36864, dtype=torch.uint8)], dim=1).cuda()
    dys = pack_blocks_cm(dy).cuda()                      # every dY block is a chunk-major image
    offs, shapes, total = ops.wgrad_layout()
    assert len(shapes) == len(JOBS)
    blob = torch.zeros(total, device="cuda")
    ops.field_wgrad(xs, dys, pts, blob)
    torch.cuda.synchronize()
    blob = blob.cpu()
    xf, dyf = x.float(), dy.float()
    for j, job in enumerate(JOBS):
        m, n = shapes[j]
        if job is None:
            assert (m, n) == ((256, 256) if j == 9 else (128, 256)) and not blob[offs[2 * j]: offs[2 * j] + m * n + m].any()
            continue
        a, mb, b, nb, has_db = job
        assert (m, n) == ((mb + (mb & 1)) * 64, nb * 64)
        m = mb * 64                                  # the rows the kernel defines (job 10: 192 of 256)
        ref = dyf[:, a * 64:(a + mb) * 64].T @ xf[:, b * 64:(b + nb) * 64]
        got = blob[offs[2 * j]: offs[2 * j] + m * n].view(m, n)
        torch.testing.assert_close(got, ref, rtol=2e-3, atol=2e-3 * float(ref.abs().max()), msg=lambda s, j=j: f"job {j}: {s}")
        if has_db:
            refb = dyf[:, a * 64:(a + mb) * 64].sum(0)
            gotb = blob[offs[2 * j + 1]: offs[2 * j + 1] + m]
            torch.testing.assert_close(gotb, refb, rtol=2e-3, atol=2e-3 * float(refb.abs().max()))
        else:
            assert offs[2 * j + 1] == -1


def test_wgrad_sums_are_the_same_from_launch_to_launch():
    """The CTAs of a job add their split-K sums into the blob in split order: repeated launches on the same stashes give
    bit-identical gradients (accumulated on top of a non-zero blob, as the passes of one backward do)."""
    g = torch.Generator().manual_seed(5)
    n_tiles = 160
    xs = torch.randint(0, 256, (n_tiles, STASH_BLOCKS * 16384 + 36864), generator=g, dtype=torch.uint8)
    xs = (xs & 0x3f).cuda()            # small finite bf16 values (high bytes < 0x40)
    dys = (torch.randint(0, 256, (n_tiles, DY_BLOCKS, 16384), generator=g, dtype=torch.uint8) & 0x3d).cuda()
    total = ops.wgrad_layout()[2]
    start = torch.randn(total, generator=g).cuda()
    blobs = []
    for _ in range(4):
        blob = start.clone()
        ops.field_wgrad(xs, dys, n_tiles * 128, blob)
        blobs.append(blob)
    torch.cuda.synchronize()
    assert torch.isfinite(blobs[0]).all() and not torch.equal(blobs[0], start)
    for b in blobs[1:]:
        assert torch.equal(b, blobs[0])


def test_wgrad_finish_derives_the_bottleneck_gradients():
    """rsn_field_wgrad_finish on a random blob against the algebra it implements (and its host mirror in ops)."""
    g = torch.Generator().manual_seed(3)
    offs, shapes, total = ops.wgrad_layout()
    blob = torch.randn(total, generator=g)
    w_b, b_b, w_m = torch.randn(256, 256, generator=g), torch.randn(256, generator=g), torch.randn(128, 290, generator=g)
    G = blob[offs[20] + 64 * 256: offs[20] + 192 * 256].view(128, 256).double()      # rows 64-191 of job 10
    dbm = blob[offs[21] + 64: offs[21] + 192].double()
    ref9 = w_m[:, 34:].double().T @ G
    ref9b = w_m[:, 34:].double().T @ dbm
    ref12 = G @ w_b.double().T + torch.outer(dbm, b_b.double())
    host, dev = blob.clone(), blob.clone().cuda()
    ops.wgrad_finish(host, w_b, b_b, w_m)
    ops.wgrad_finish(dev, w_b.cuda(), b_b.cuda(), w_m.cuda())
    torch.cuda.synchronize()
    for got in (host, dev.cpu()):
        torch.testing.assert_close(got[offs[18]: offs[18] + 65536].view(256, 256).double(), ref9, rtol=1e-4, atol=1e-3)
        torch.testing.assert_close(got[offs[19]: offs[19] + 256].double(), ref9b, rtol=1e-4, atol=1e-3)
        torch.testing.assert_close(got[offs[24]: offs[24] + 32768].view(128, 256).double(), ref12, rtol=1e-4, atol=1e-3)
        torch.testing.assert_close(got[offs[25]: offs[25] + 128].double(), dbm)
        untouched = torch.ones(total, dtype=torch.bool)
        untouched[offs[18]: offs[19] + 256] = False
        untouched[offs[24]: offs[25] + 128] = False
        assert torch.equal(got[untouched], blob[untouched])
