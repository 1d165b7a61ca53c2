"""Generate tests/golden/loader_golden.npz: what the REFERENCE's own `StereoHumanDataset` (lib/human_loader.py) reads
from the synthetic dataset that gps_gaussian_b200.synth_dataset writes.

    python tests/golden/make_loader_golden.py <GPS-Gaussian checkout>

Stores, for sample 0 at 96^2 (train phase, novel view 3), the source views' rectified image, flow, valid mask and
calibration as the loader returns them, the novel view's shape, and the test-phase item's calibration shapes -- plus the
written depth maps and camera matrices the loader consumed, so the test can check that the writer still writes them."""
import os
import sys
import tempfile
from types import SimpleNamespace

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
RES = 96


def main(ref):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, ref)
    from gps_gaussian_b200 import synth_dataset
    from lib.human_loader import StereoHumanDataset
    out = {}
    with tempfile.TemporaryDirectory() as root:
        names = synth_dataset.write_dataset(root, n_train=2, n_val=1, res=RES, hr=True)
        opt = SimpleNamespace(data_root=root, test_data_root=None, use_processed_data=False, source_id=[0, 1],
                              train_novel_id=[2, 3, 4], val_novel_id=[3], src_res=RES, use_hr_img=True, bg_color=[0, 0, 0],
                              znear=0.01, zfar=100.0, trans=[0.0, 0.0, 0.0], scale=1.0)
        ds = StereoHumanDataset(opt, phase="train")
        out["sample_list"] = np.array(ds.sample_list)
        out["train_names"] = np.array(names["train"])
        item = ds.get_item(0, novel_id=[3])
        for v in ("lmain", "rmain"):
            for k in ("img", "mask", "flow", "valid", "intr", "extr", "ref_intr", "Tf_x"):
                out[f"{v}_{k}"] = item[v][k].numpy()
        out["novel_img_shape"] = np.array(item["novel_view"]["img"].shape)
        out["novel_width"] = np.array(int(item["novel_view"]["width"]))
        opt.test_data_root = os.path.join(root, "val")
        t = StereoHumanDataset(opt, phase="test").get_test_item(0, source_id=[0, 1])
        out["test_lmain_intr_ori_shape"] = np.array(t["lmain"]["intr_ori"].shape)
        out["test_rmain_extr_ori_shape"] = np.array(t["rmain"]["extr_ori"].shape)
        out["test_novel_height"] = np.array(int(t["novel_view"]["height"]))
        base = os.path.join(root, "train")
        for vid in (0, 1):
            out[f"written_depth_{vid}"] = cv2.imread(os.path.join(base, "depth", names["train"][0], f"{vid}.png"), -1)
            out[f"written_intrinsic_{vid}"] = np.load(os.path.join(base, "parm", names["train"][0], f"{vid}_intrinsic.npy"))
            out[f"written_extrinsic_{vid}"] = np.load(os.path.join(base, "parm", names["train"][0], f"{vid}_extrinsic.npy"))
    np.savez_compressed(os.path.join(HERE, "loader_golden.npz"), **out)


if __name__ == "__main__":
    main(sys.argv[1])
