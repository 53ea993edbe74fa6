"""Drop-in check of the YAML grammar against the reference's own model zoo (fixture: tests/golden/make_golden.py zoo, the parsed
layer tables keyed by their path below the reference's cfg/models).  Every stock detection YAML whose module set is registered here
must construct - the one known exception asks for scene-aware MoT routing, which raises by design (DESIGN.md §7)."""
import json
import os

from _util import GOLD


def test_stock_detection_yamls_construct():
    from yolo_master_b200.nn import tasks
    supported = set(tasks.MODULES) | set(tasks.MIXTURE_MODULES) | {"nn.Upsample"}
    zoo = json.load(open(os.path.join(GOLD, "zoo.golden.json")))
    files = sorted(zoo)
    other = [f for f in files if any(f"/{t}/" in f for t in ("seg", "pose", "obb", "cls")) and f.endswith("-n.yaml")]
    files = [f for f in files if "/det/" in f or f.startswith("26/") or "/exp/" in f]
    built, skipped, raised = 0, 0, []
    for f in files:
        d = zoo[f]
        if {layer[2] for layer in d.get("backbone", []) + d.get("head", [])} - supported:
            skipped += 1                                          # a module family that is not on the B200 path (DESIGN.md §8)
            continue
        if not f.endswith("-n.yaml") and not f.endswith("-p2.yaml") and "/exp/" not in f and not f.startswith("26/"):
            continue                                              # one scale per family keeps the CPU suite short
        try:
            tasks.DetectionModel(d)
            built += 1
        except NotImplementedError as e:
            raised.append((f, str(e)))
    for f in other:                                               # the n file of every seg / pose / obb / cls zoo constructs too
        d = zoo[f]
        if not ({layer[2] for layer in d.get("backbone", []) + d.get("head", [])} - supported):
            tasks.DetectionModel(d)
            built += 1
    assert built >= 60, (built, skipped)
    assert [r[0] for r in raised] == ["master/v0_10/det/yolo-master-mot-scene-n.yaml"], raised
    assert skipped <= 3, skipped                                  # 102 detection YAMLs in the zoo, 99 on the path
