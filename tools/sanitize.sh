#!/bin/bash
# GPU box: compute-sanitizer over a small end-to-end run of the chain (all seven kernels + the depth path).
#   bash tools/sanitize.sh <tag>
TAG=${1:-san}; OUT=gpurun_out/$TAG; mkdir -p $OUT
cat > /tmp/san_run.py <<'P'
import sys, numpy as np
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import helpers, stair_step_detector_b200 as S
W, H = 640, 480
cfg = S.default_config(W, H)
base = S.default_scene(W, H, noise_sigma=0.0025, dropout=0.03, n_holes=3)
xf = S.scene_transform(base)
scenes = [S.randomize_scene(base, 7, i, 3, 8) for i in range(6)]
depth = np.stack([S.synth_depth_host(sc) for sc in scenes])
xyz = np.stack([S.deproject_host(sc, d) for sc, d in zip(scenes, depth)])
orc = helpers.load_oracle()
with S.Detector(cfg, xf, max_frames=len(scenes)) as det:
    det.set_overlay(S.inverse3(xf.a), S.scene_intrinsics(base))  # drawStairStep projection in k_finalize
    det.process_host(xyz)
    assert len(det.overlay(0)) == len(det.steps(0)[0])
    a = [det.steps(f)[0] for f in range(len(scenes))]
    labels = [det.labels(f) for f in range(len(scenes))]
    det.process_depth_host(depth, S.scene_intrinsics(base))
    b = [det.steps(f)[0] for f in range(len(scenes))]
    det.set_vertical_faces(True)  # k_riser_reduce
    det.process_host(xyz)
    ris = [det.vertical_faces(f) for f in range(len(scenes))]
    det.process_depth_host(depth, S.scene_intrinsics(base))
    assert ris == [det.vertical_faces(f) for f in range(len(scenes))]
for f in range(len(scenes)):
    assert ris[f] == helpers.oracle_vertical_faces(orc, cfg, xf, xyz[f].reshape(-1, 3))
for f in range(len(scenes)):
    o = helpers.oracle_process(orc, cfg, xf, xyz[f])
    assert np.array_equal(labels[f], o.labels) and len(a[f]) == len(o.steps) == len(b[f])
# the large frame-size class (k_outline<OutlineShared>: 512-thread blocks, pruned line fits, per-thread distance arrays)
W2, H2 = 1600, 1200
cfg2 = S.default_config(W2, H2)
base2 = S.default_scene(W2, H2, noise_sigma=0.0025, dropout=0.03, n_holes=3)
xf2 = S.scene_transform(base2)
sc2 = [S.randomize_scene(base2, 11, i, 3, 8) for i in range(2)]
xyz2 = np.stack([S.deproject_host(sc, S.synth_depth_host(sc)) for sc in sc2])
with S.Detector(cfg2, xf2, max_frames=2) as det:
    det.process_host(xyz2)
    c = [det.steps(f)[0] for f in range(2)]
    lab2 = [det.labels(f) for f in range(2)]
for f in range(2):
    o = helpers.oracle_process(orc, cfg2, xf2, xyz2[f])
    assert np.array_equal(lab2[f], o.labels) and len(c[f]) == len(o.steps)
    for (h, q), s in zip(c[f], o.steps):
        assert abs(h - s["height"]) < 1e-4 and np.abs(q - s["quad"]).max() < 1e-4
print("sanitizer run ok:", [len(x) for x in a], [len(x) for x in c])
P
for tool in memcheck racecheck synccheck initcheck; do
  echo "== $tool"
  timeout 900 compute-sanitizer --tool $tool --print-limit 20 python /tmp/san_run.py > $OUT/$tool.log 2>&1
  tail -4 $OUT/$tool.log
done
