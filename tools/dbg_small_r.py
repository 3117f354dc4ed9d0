import sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / 'tests'))
from dynamicslamtool_b200 import MovingObjectRemoval, Synth, load_product
from helpers import write_cfg
import tempfile
cfg = write_cfg(tempfile.mkdtemp(), base=ROOT / 'config' / 'MOR_config_hdl64.txt', ec_distance_threshold=0.11, min_cluster_size=20)
s = Synth(2, 2)
m = MovingObjectRemoval(cfg, 4, 3, binding=load_product(), max_points=s.max_points)
for f in range(int(sys.argv[1]) if len(sys.argv) > 1 else 3):
    pts, pose = s.frame(f)
    m.push_raw_cloud_and_pose(pts, pose); m.filter_cloud()
    print(f, m.counts(), flush=True)
