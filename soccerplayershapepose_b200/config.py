"""Constants of the SMPL hot path that the reference keeps in `PlayerReconstruction/config.py`.

Only what the hot path needs (SURVEY.md section 2, row "config.py (joint-map part)"): the
default data locations used by `load_smpl_model`, the two camera constants, and the integer
joint-index tables.  The index tables are pure integer data and must stay bit-exact with the
reference (`config.py:29-38`); `tests/test_oracle.py::test_index_tables_bit_exact` checks them against golden
vectors generated from the reference file itself.
"""
import os

_ADDITIONAL = os.environ.get("B200SMPL_ADDITIONAL_DIR", os.path.join("PlayerReconstruction", "additional"))

# data locations (reference config.py:3-8; the directory is not part of the reference tree)
SMPL_MODEL_DIR = os.path.join(_ADDITIONAL, "smpl")
SMPL_FACES_PATH = os.path.join(_ADDITIONAL, "smpl_faces.npy")
SMPL_MEAN_PARAMS_PATH = os.path.join(_ADDITIONAL, "neutral_smpl_mean_params_6dpose.npz")
J_REGRESSOR_EXTRA_PATH = os.path.join(_ADDITIONAL, "J_regressor_extra.npy")
COCOPLUS_REGRESSOR_PATH = os.path.join(_ADDITIONAL, "cocoplus_regressor.npy")
H36M_REGRESSOR_PATH = os.path.join(_ADDITIONAL, "J_regressor_h36m.npy")

# camera constants (reference config.py:15-16)
FOCAL_LENGTH = 5000.0
REGRESSOR_IMG_WH = 256

# layout of the 90-joint superset returned by SMPL.forward (reference config.py:19-30 comment,
# models/smpl_official.py:30-34): [0:24] SMPL chain joints, [24:45] vertex-picked face / feet /
# finger-tip joints, [45:54] "extra" regressor, [54:73] COCO-plus regressor, [73:90] H36M regressor
NUM_SMPL_JOINTS = 24
NUM_VERTEX_JOINTS = 21
NUM_EXTRA_JOINTS = 9
NUM_COCOPLUS_JOINTS = 19
NUM_H36M_JOINTS = 17
NUM_ALL_JOINTS = NUM_SMPL_JOINTS + NUM_VERTEX_JOINTS + NUM_EXTRA_JOINTS + NUM_COCOPLUS_JOINTS + NUM_H36M_JOINTS

# 17 COCO keypoints out of the superset: nose, l-eye, r-eye, l-ear, r-ear, then shoulders,
# elbows, wrists, hips, knees, ankles (left before right)
ALL_JOINTS_TO_COCO_MAP = [24, 26, 25, 28, 27, 16, 17, 18, 19, 20, 21, 1, 2, 4, 5, 7, 8]
# the H36M block is the tail of the superset
ALL_JOINTS_TO_H36M_MAP = list(range(NUM_ALL_JOINTS - NUM_H36M_JOINTS, NUM_ALL_JOINTS))
# 17 -> LSP-17 / LSP-14 re-ordering of the H36M block
H36M_TO_J17 = [6, 5, 4, 1, 2, 3, 16, 15, 14, 11, 12, 13, 8, 10, 0, 7, 9]
H36M_TO_J14 = H36M_TO_J17[:14]
# the LSP-14 joints of the superset, joints[:, ALL_JOINTS_TO_H36M_MAP][:, H36M_TO_J14] (the MPJPE joints)
ALL_JOINTS_TO_J14_MAP = [ALL_JOINTS_TO_H36M_MAP[i] for i in H36M_TO_J14]
# Keypoint-RCNN order is the COCO order
SMPL_TO_KPRCNN_MAP = list(ALL_JOINTS_TO_COCO_MAP)

# body_pose joints (0-based inside the 23 body joints) frozen by the fitting loops
# (player_recon.py:1175-1177, 1202-1206): ankles 6,7 and hands 21,22
FITTING_FROZEN_BODY_JOINTS = [6, 7, 21, 22]
