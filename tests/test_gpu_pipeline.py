"""GPU: the batched device-resident Pipeline (preprocess -> detect -> pose) vs the per-frame oracle chain, plus
size-independent properties at the full 4K size (BASELINE.json configs 2-4)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pipe(camera, lut, dictionary, ref_params):
    import apse_uav_b200 as A
    K, D = camera
    p = A.Pipeline(K, D, (3840, 2160), lut, dictionary, ref_params, max_batch=6, max_markers=256)
    yield p
    p.engine.close()


def test_pipeline_matches_oracle_chain(pipe, oracle, camera, lut, dictionary, ref_params, frames4k):
    import torch
    import apse_uav_b200 as A
    K, D = camera
    ox, oy = oracle.init_undistort_map(K, D, 3840, 2160)
    frames = [frames4k["sparse"], frames4k["dense"]]
    res = A.Pipeline.to_host(pipe.run(torch.from_numpy(np.stack(frames)).cuda()))
    for i, f in enumerate(frames):
        _, gray = oracle.preprocess(f, ox, oy, lut)
        oc, oi, _ = oracle.detect_markers_apriltag(gray, dictionary.raw, ref_params)
        orv, otv = oracle.estimate_pose_single_markers(oc, 0.55, K, D)
        n = int(res["n"][i])
        assert n == len(oi) and np.array_equal(res["ids"][i, :n], oi)
        assert np.abs(res["corners"][i, :n] - oc).max() <= 1e-3
        assert (np.linalg.norm(res["tvec"][i, :n] - otv[:, 0], axis=-1) / np.linalg.norm(otv[:, 0], axis=-1)).max() < 1e-4
        assert (np.linalg.norm(res["rvec"][i, :n] - orv[:, 0], axis=-1) / np.linalg.norm(orv[:, 0], axis=-1)).max() < 1e-4


def test_sequence_properties_full_size(pipe, dictionary, frames4k):
    """14 frames > max_batch (chunking), translated copies of one frame: every frame finds the same ids, corners
    move by the translation (away from the border, where undistortion is locally a shift-invariant warp only
    approximately -> 2 px bound), results independent of the position inside the batch, launches are counted."""
    import torch
    import apse_uav_b200 as A
    base = torch.from_numpy(frames4k["sparse"]).cuda()
    shifts = [(0, 0), (3, 5), (0, 0), (-4, 2), (7, -6), (0, 0), (1, 1), (0, 0), (2, -3), (-5, -5), (0, 0), (4, 4), (6, 0), (0, 0)]
    seq = torch.stack([torch.roll(base, shifts=(dy, dx), dims=(0, 1)) for dx, dy in shifts])
    l0 = pipe.launches
    res = A.Pipeline.to_host(pipe.run(seq))
    assert pipe.launches - l0 >= 3 * 12      # 3 batches x (1 preprocess + 10 detect + 1 decode + 1 pose)
    n0 = int(res["n"][0])
    assert n0 >= 4
    ref_ids = res["ids"][0, :n0]
    zero = [i for i, s in enumerate(shifts) if s == (0, 0)]
    for i in zero:   # identical frames -> bit-identical results wherever they sit in a batch
        assert np.array_equal(res["ids"][i], res["ids"][0]) and np.array_equal(res["corners"][i], res["corners"][0])
        assert np.array_equal(res["tvec"][i, :n0], res["tvec"][0, :n0])
    for i, (dx, dy) in enumerate(shifts):
        n = int(res["n"][i])
        assert sorted(res["ids"][i, :n].tolist()) == sorted(ref_ids.tolist())
        for m in range(n):
            j = list(ref_ids).index(res["ids"][i, m])
            d = res["corners"][i, m] - res["corners"][0, j] - np.float32([dx, dy])
            assert np.abs(d).max() < 2.0
    # pose sanity: tvec_z within the 15-60 m band the synthetic marker sizes imply
    assert ((res["tvec"][0, :n0, 2] > 10) & (res["tvec"][0, :n0, 2] < 80)).all()


def _golden_frames(dictionary, name):
    import torch
    from conftest import golden_csv, golden_events
    from tools import synth
    g, ref = golden_csv(name)
    frames = np.stack(list(synth.make_sequence(dictionary.bytesList, g["base_seed"], g["n_frames"], leds=g["leds"], events=golden_events(g))))
    return g, ref, torch.from_numpy(frames).cuda()


def test_sequence_csv_matches_reference_script(pipe, dictionary):
    """End to end on the GPU: frames -> Pipeline -> native two-pass post-pass (csrc/sequence.cu) -> CSV rows of
    aruco_detect.py:146-185, compared with the rows the reference script itself wrote for the same seeded frames
    (tests/golden/sequence_4k.json), and with the per-frame Python mirror of the loop (identical rows and CSV text)."""
    pytest.importorskip("cv2")   # tools.synth renders the frames with cv2.warpPerspective / resize
    from conftest import assert_csv_rows_match
    from apse_uav_b200 import shard, sequence
    g, ref, frames = _golden_frames(dictionary, "sequence_4k.json")
    rows = shard.run_sequence(pipe, frames, as_rows=True)
    assert_csv_rows_match(sequence.rows_to_dicts(rows), ref)
    mirror = shard.run_sequence_python(pipe, frames)
    assert sequence.rows_to_dicts(rows) == mirror
    assert sequence.rows_to_csv(rows) == shard.rows_to_csv(mirror)


def test_events_sequence_matches_reference_script(pipe, dictionary):
    """64 frames with vanishing / returning / jumping markers and an empty frame (tests/golden/sequence_4k_events.json): the
    gating and relabel branches of aruco_detect.py:613,637,669, the altitude fallback :639-642, every stale CSV value and the
    LED read-out, native post-pass vs the reference script's rows and vs the Python mirror."""
    pytest.importorskip("cv2")
    from conftest import assert_csv_rows_match
    from apse_uav_b200 import shard, sequence
    g, ref, frames = _golden_frames(dictionary, "sequence_4k_events.json")
    rows = shard.run_sequence(pipe, frames, leds=True, as_rows=True)
    assert_csv_rows_match(sequence.rows_to_dicts(rows), ref)
    assert sequence.rows_to_dicts(rows) == shard.run_sequence_python(pipe, frames, leds=True)


def test_reference_script_runs_with_import_swap(dictionary, tmp_path):
    """north_star: "aruco_detect.py runs with only an import swap".  The reference's own script text (compiled from where it
    lies by oracle/build_ref.py, lines 1-2 swapped to apse_uav_b200, user paths redirected) is executed on the GPU and its
    CSV is compared with the CSV the same text produced on cv2 (tests/golden/sequence_4k.json)."""
    cv2 = pytest.importorskip("cv2")
    from conftest import GOLDEN, assert_csv_rows_match, golden_csv
    from tools import synth, run_reference_script
    if not run_reference_script.available("apse"):
        pytest.skip("oracle/_ref/aruco_detect.swap.bin not built: needs the reference's aruco_detect.py, which is not part of this repository")
    g, ref = golden_csv("sequence_4k.json")
    img = tmp_path / "frames"
    img.mkdir()
    for k, f in enumerate(synth.make_sequence(dictionary.bytesList, g["base_seed"], g["n_frames"])):
        cv2.imwrite(str(img / ("image_%04d.png" % (k + 1))), f)
    csv = run_reference_script.run(str(img), str(tmp_path / "out.csv"), GOLDEN, module="apse")
    lines = csv.splitlines()
    assert lines[0] == g["csv"][0]
    got = np.array([[float(v) for v in line.split(",")] for line in lines[1:]])
    assert_csv_rows_match(got, ref)


def test_sharded_sequence_world2(dictionary, tmp_path):
    """BASELINE.json configs[3]: the same sequence frame-sharded over two GPUs (one process per GPU, NCCL only for the
    gather of the per-frame results and the LED job exchange) gives the rows of the single-GPU run."""
    import subprocess, sys, torch
    pytest.importorskip("cv2")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from conftest import ROOT
    script = tmp_path / "worker.py"
    script.write_text(WORLD2_WORKER)
    out = tmp_path / "rows.json"
    port = str(29700 + __import__("os").getpid() % 200)
    rc = subprocess.call([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", port, str(script), ROOT, str(out)], timeout=900)
    assert rc == 0
    import json
    res = json.load(open(out))
    assert res["sharded"] == res["single"]
    assert res["rounds"] >= 5 and res["streamed"] == res["single_noleds"]
    from conftest import assert_csv_rows_match, golden_csv
    assert_csv_rows_match(res["sharded"], golden_csv("sequence_4k_events.json")[1])


WORLD2_WORKER = r"""
import json, os, sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import numpy as np, torch, torch.distributed as dist
import apse_uav_b200 as A
from apse_uav_b200 import aruco, shard
from tools import synth
import __graft_entry__ as G
from conftest import golden_csv, golden_events
rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
cam = json.load(open(os.path.join(sys.argv[1], "tests", "golden", "cam_params.json")))
K, D = np.array(cam["mtx"]), np.array(cam["dist"]).ravel()
d = aruco.getPredefinedDictionary(aruco.DICT_4X4_50)
g, _ = golden_csv("sequence_4k_events.json")
frames = np.stack(list(synth.make_sequence(d.bytesList, g["base_seed"], g["n_frames"], leds=g["leds"], events=golden_events(g))))
pipe = A.Pipeline(K, D, (3840, 2160), G.gamma_lut(), d, G.reference_parameters(aruco), max_batch=6, device=lr, max_markers=64, streams=3)
lo, hi = shard.shard_bounds(len(frames), world)[rank]
rows = shard.run_sequence(pipe, torch.from_numpy(frames[lo:hi]).cuda(), rank, world, leds=True)
# the streamed run: frames dealt out in rounds, post-pass of round k on rank 0 while both ranks compute round k + 1
plan = shard.round_plan(len(frames), world, 6, tail=2)
mine = np.concatenate([frames[a:b] for rnd in plan for a, b in [rnd[rank]]])
streamed = None
for _ in range(2):   # twice: the second run reuses the cached buffers
    streamed = shard.run_sequence_streamed(pipe, torch.from_numpy(mine).cuda(), plan, rank, world, chunk_frames=12)
if rank == 0:
    single = shard.run_sequence(pipe, torch.from_numpy(frames).cuda(), 0, 1, leds=True)
    single_noleds = shard.run_sequence(pipe, torch.from_numpy(frames).cuda(), 0, 1)
    json.dump({"sharded": rows, "single": single, "streamed": streamed, "single_noleds": single_noleds, "rounds": len(plan)}, open(sys.argv[2], "w"))
dist.barrier()
dist.destroy_process_group()
"""


@pytest.mark.parametrize("streams", [0, 3])
def test_streamed_sequence_equals_plain(camera, lut, dictionary, ref_params, streams):
    """shard.run_sequence_streamed (frames dealt out in rounds, post-pass fed chunk by chunk behind the pipeline: what bench.py
    times) gives the rows and the CSV text of shard.run_sequence on the 64-frame events sequence, for several round / chunk sizes."""
    pytest.importorskip("cv2")
    import torch
    import apse_uav_b200 as A
    from apse_uav_b200 import shard, sequence
    K, D = camera
    pipe = A.Pipeline(K, D, (3840, 2160), lut, dictionary, ref_params, max_batch=6, max_markers=64, streams=streams)
    g, ref, frames = _golden_frames(dictionary, "sequence_4k_events.json")
    want = sequence.rows_to_csv(shard.run_sequence(pipe, frames, as_rows=True))
    for batch, tail, chunk in ((6, 2, 12), (6, 0, 1), (5, 1, 1000), (6, 2, 12)):
        plan = shard.round_plan(len(frames), 1, batch, tail=tail)
        rows = shard.run_sequence_streamed(pipe, frames, plan, as_rows=True, chunk_frames=chunk)
        assert len(rows) == len(frames) and sequence.rows_to_csv(rows) == want
    pipe.close()


def test_multi_stream_equals_single_stream(pipe, camera, lut, dictionary, ref_params, frames4k):
    """sub-batches in flight on several streams / contexts give bit-identical results."""
    import torch
    import apse_uav_b200 as A
    K, D = camera
    p3 = A.Pipeline(K, D, (3840, 2160), lut, dictionary, ref_params, max_batch=5, max_markers=256, streams=3, ring=6)
    frames = torch.from_numpy(np.stack([frames4k["sparse"], frames4k["dense"], frames4k["sparse"], frames4k["dense"], frames4k["sparse"]])).cuda()
    a = A.Pipeline.to_host(p3.run_batch(frames, want_rejected=True))
    b = A.Pipeline.to_host(pipe.run_batch(frames, want_rejected=True))
    for k in ("n", "ids", "corners", "n_rejected", "rejected", "rvec", "tvec"):
        assert np.array_equal(a[k], b[k]), k
    # overlapped mode: results are waited for later; consecutive batches share contexts and staging buffers
    frames2 = torch.roll(frames, shifts=(5, 3), dims=(1, 2))
    pending = [p3.run_batch(f, want_rejected=True, sync=False, input_ready=True) for f in (frames, frames2, frames, frames2, frames)]
    outs = [A.Pipeline.to_host(d) for d in pending]
    b2 = A.Pipeline.to_host(pipe.run_batch(frames2, want_rejected=True))
    for o, ref in zip(outs, (b, b2, b, b2, b)):
        for k in ("n", "ids", "corners", "n_rejected", "rejected", "rvec", "tvec"):
            assert np.array_equal(o[k], ref[k]), k
    p3.close()


def test_host_stream_equals_device_batches(pipe, frames4k):
    """end-to-end host path (double-buffered H2D overlapped with compute) returns what run_batch returns"""
    import torch
    f = torch.from_numpy(np.stack([frames4k["sparse"], frames4k["dense"], frames4k["sparse"]]))
    host = [f[:2].clone().pin_memory(), f[1:].clone().pin_memory(), f[:1].clone().pin_memory()]
    outs = list(pipe.run_host_stream(host))
    assert len(outs) == 3
    for hb, o in zip(host, outs):
        ref = pipe.to_host(pipe.run_batch(hb.cuda()))
        for k in ("n", "ids", "corners", "rvec", "tvec"):
            assert np.array_equal(o[k], ref[k]), k


def test_patch_sums_numpy_slicing(pipe):
    """LED read-out kernel = np.sum(gray[y-2:y+3, x-2:x+3]) including numpy's negative-start / clamped-stop slicing"""
    import torch
    rng = np.random.default_rng(9)
    gray = rng.integers(0, 256, (2, 37, 53), dtype=np.uint8)
    pts = [(f, x, y) for f in (0, 1) for x in (0, 1, 2, 3, 25, 49, 50, 51, 52, 53, 60) for y in (0, 1, 2, 17, 33, 34, 35, 36, 37, 40)]
    got = pipe.engine.patch_sums(torch.from_numpy(gray).cuda(), pts, half=2)
    ref = [int(np.sum(gray[f][y - 2:y + 3, x - 2:x + 3])) for f, x, y in pts]
    assert got.tolist() == ref


def test_sequence_with_leds_matches_reference_script(pipe, dictionary):
    """SURVEY.md 8f-1: frames with a rendered LED strip -> leds_ID column of the reference script's CSV"""
    pytest.importorskip("cv2")
    from conftest import assert_csv_rows_match
    from apse_uav_b200 import shard
    g, ref, frames = _golden_frames(dictionary, "sequence_4k_leds.json")
    rows = shard.run_sequence(pipe, frames, leds=True)
    assert_csv_rows_match(rows, ref)
    assert [r["leds_ID"] for r in rows] == g["leds"]
    assert rows == shard.run_sequence_python(pipe, frames, leds=True)


def test_multi_stream_gray_equals_single_stream(pipe, camera, lut, dictionary, ref_params, frames4k):
    """want_gray / gray_out with sub-batches on several streams: the returned gray frames are complete (the current stream is
    ordered behind the preprocess streams before they are concatenated) and equal the single-stream ones."""
    import torch
    import apse_uav_b200 as A
    K, D = camera
    p3 = A.Pipeline(K, D, (3840, 2160), lut, dictionary, ref_params, max_batch=5, max_markers=256, streams=3, ring=6)
    frames = torch.from_numpy(np.stack([frames4k["sparse"], frames4k["dense"], frames4k["sparse"], frames4k["dense"], frames4k["sparse"]])).cuda()
    ref = pipe.run_batch(frames, want_gray=True)["gray"]
    for _ in range(3):
        got = p3.run_batch(frames, want_gray=True)["gray"]
        assert torch.equal(got, ref)
    seq_gray = torch.zeros((10, 2160, 3840), dtype=torch.uint8, device="cuda")
    det = p3.run_sequence(torch.cat([frames, frames]), gray_out=seq_gray)
    torch.cuda.synchronize()
    assert torch.equal(seq_gray[:5], ref) and torch.equal(seq_gray[5:], ref)
    one = A.Pipeline.to_host(pipe.run_batch(frames))
    for k in ("n", "ids", "corners", "rvec", "tvec"):
        assert np.array_equal(det[k][:5].cpu().numpy(), one[k]) and np.array_equal(det[k][5:].cpu().numpy(), one[k]), k
    p3.close()
