import sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / 'tests'))
from dynamicslamtool_b200 import MovingObjectRemoval, Synth, load_product
s = Synth(2, 2)
m = MovingObjectRemoval(ROOT / 'config' / 'MOR_config_hdl64.txt', 4, 3, binding=load_product(), max_points=s.max_points)
for f in range(0, 108):
    pts, pose = s.frame(f)
    try:
        m.push_raw_cloud_and_pose(pts, pose); m.filter_cloud()
        c = m.counts()
    except Exception as e:
        print("FAIL at frame", f, e); break
    if f > 55: print(f, c["NC"], c["K"], c["ERRFLAGS"], flush=True)
