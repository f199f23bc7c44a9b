"""On-disk formats and episode iteration of the reference (SURVEY 8b 'On-disk state', 8f rank 2) - host side only.

Dataset names are the reference's, typos included, so files written by either side load in the other:
  memory_data/<seq>.h5   memory_features f32 (cells,256) | proj_indices i32 (T,480,640,1) | semmap_gt i32 (cells,)
                         (SMNet/build_memory_data.py:150-153)
  sensor_data/<seq>.h5   rgb, depth, projection_indices f32 (T,480,640,3) [world xyz], masks_outliers, sensor_positions,
                         detection_data, segmentation_data (SMNet/build_data.py:275-286)
  <out>/memory/<seq>     semmap i32 (cells,) | impicit_memory [sic] f32 (cells,512) | observations f32 (cells,)
                         (detic/modeling/meta_arch/custom_rcnn.py:527-530; re-read by SMNet/loader.py:216-223)
  <out>/heightmax/<seq>  state f32 (cells,C) | observed u8 (cells,) | height_map f32 (cells,): the SMNet encoder's map after the
                         episode's last frame, what its decoder takes (EpisodeRunner(regime="heightmax"))
Containers: HDF5 through h5py when it is importable (it is not in this image), otherwise ``.npz`` with the same
keys.  ``open_store`` picks by what exists on disk; a missing or unreadable file RAISES (the reference's silent
zero-memory fallback, loader.py:208-211, is deliberately not reproduced).
"""
from __future__ import annotations

import math
import os
from typing import Dict, Iterator, List, Optional, Sequence, Tuple

import numpy as np

try:                                    # optional: HDF5 container
    import h5py                         # type: ignore
except Exception:                       # pragma: no cover - h5py is absent in this image
    h5py = None

MEMORY_KEYS = ("memory_features", "proj_indices", "semmap_gt")
SAVED_MEMORY_KEYS = ("semmap", "impicit_memory", "observations")        # sic: custom_rcnn.py:528


class StoreError(IOError):
    pass


def _candidates(path: str) -> List[str]:
    base, ext = os.path.splitext(path)
    if ext in (".h5", ".npz"):
        return [path, base + (".npz" if ext == ".h5" else ".h5")]
    return [path, path + ".h5", path + ".npz"]


def open_store(path: str) -> Dict[str, np.ndarray]:
    """Read every dataset of an HDF5 / npz store into a dict of numpy arrays (files here are tens of MB)."""
    for p in _candidates(path):
        if not os.path.isfile(p):
            continue
        with open(p, "rb") as f:
            magic = f.read(8)
        if magic.startswith(b"\x89HDF"):
            if h5py is None:
                raise StoreError(f"{p} is HDF5 but h5py is not installed; convert it to .npz with the same dataset names")
            with h5py.File(p, "r") as h:
                return {k: np.array(h[k]) for k in h.keys()}
        if magic.startswith(b"PK"):
            with np.load(p, allow_pickle=False) as z:
                return {k: z[k] for k in z.files}
        raise StoreError(f"{p}: neither HDF5 nor npz")
    raise StoreError(f"no store at {path} (tried {', '.join(_candidates(path))})")


def write_store(path: str, arrays: Dict[str, np.ndarray], container: Optional[str] = None) -> str:
    """Write a store; container 'h5' | 'npz' | None (h5 when h5py exists and the name does not end in .npz)."""
    if container is None:
        container = "npz" if (h5py is None or path.endswith(".npz")) else "h5"
    os.makedirs(os.path.dirname(os.path.abspath(path)) or ".", exist_ok=True)
    if container == "h5":
        if h5py is None:
            raise StoreError("h5py is not installed")
        with h5py.File(path, "w") as h:
            for k, v in arrays.items():
                h.create_dataset(k, data=v, dtype=v.dtype)
        return path
    out = path if path.endswith(".npz") else os.path.splitext(path)[0] + ".npz"
    with open(out, "wb") as f:
        np.savez(f, **arrays)
    return out


# ---- saved memory (custom_rcnn.py:518-530 <-> loader.py:216-223) ---------------------------------------------------
def save_memory(path: str, semmap, implicit_memory, observations, container: Optional[str] = None) -> str:
    """{semmap int32 (cells,), impicit_memory float32 (cells,C), observations float32 (cells,)}.  Tensors are moved to
    the host here - this is the one D2H of the grid, once per sequence (the reference does it at frame 0, :521)."""
    to_np = lambda t: t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
    return write_store(path, {"semmap": to_np(semmap).astype(np.int32), "impicit_memory": to_np(implicit_memory).astype(np.float32),
                              "observations": to_np(observations).astype(np.float32)}, container)


def load_memory(path: str) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """-> (semmap + 1 [empty space -1 -> 0, loader.py:221], implicit_memory, observations)."""
    d = open_store(path)
    missing = [k for k in SAVED_MEMORY_KEYS if k not in d]
    if missing:
        raise StoreError(f"{path}: missing datasets {missing}")
    return d["semmap"] + 1, d["impicit_memory"], d["observations"]


# ---- height-max memory after an episode's last frame -------------------------------------------------------------
HEIGHTMAX_KEYS = ("state", "observed", "height_map")


def save_heightmax(path: str, state, observed, height_map, container: Optional[str] = None) -> str:
    """{state float32 (cells,C), observed uint8 (cells,), height_map float32 (cells,)}; tensors are moved to the host here."""
    to_np = lambda t: t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
    return write_store(path, {"state": to_np(state).astype(np.float32), "observed": to_np(observed).astype(np.uint8),
                              "height_map": to_np(height_map).astype(np.float32)}, container)


def load_heightmax(path: str) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """-> (state, observed, height_map) as save_heightmax wrote them."""
    d = open_store(path)
    missing = [k for k in HEIGHTMAX_KEYS if k not in d]
    if missing:
        raise StoreError(f"{path}: missing datasets {missing}")
    return d["state"], d["observed"], d["height_map"]


# ---- memory_data (build_memory_data.py:108-153) ------------------------------------------------------------------
def map_dims_from_info(semmap_info: dict, env: str, res_downsample: int = 10) -> Tuple[int, int, np.ndarray]:
    """(map_width, map_height, map_world_shift) as build_memory_data.py:108-115 derives them."""
    dim = semmap_info[env]["dim"]
    return math.ceil(dim[0] / res_downsample), math.ceil(dim[2] / res_downsample), np.asarray(semmap_info[env]["map_world_shift"], np.float32)


def write_memory_data(path: str, proj_indices: np.ndarray, n_cells: int, feat_dim: int = 256, semmap_gt: Optional[np.ndarray] = None,
                      container: Optional[str] = None) -> str:
    """memory_features zeros (cells,256) f32, proj_indices (T,H,W,1) i32, semmap_gt zeros (cells,) i32 (:147-153)."""
    pi = np.asarray(proj_indices)
    if pi.ndim == 3:
        pi = pi[..., None]
    return write_store(path, {"memory_features": np.zeros((n_cells, feat_dim), np.float32), "proj_indices": pi.astype(np.int32),
                              "semmap_gt": (np.zeros(n_cells) if semmap_gt is None else semmap_gt).astype(np.int32)}, container)


# ---- episode ordering and reset flags (loader.py:97-117, 289-293) -----------------------------------------------
def sequence_sort_key(name: str) -> Tuple[str, int]:
    """loader.py:97-105: (scene prefix incl. trailing '_', integer sequence id)."""
    parts = name.split("_")
    return "".join(p + "_" for p in parts[:-1]), int(parts[-1].split(".")[0])


def order_files(files: Sequence[str], test_type: str = "default") -> List[str]:
    """Sorted episode files; 'longterm' replays every chunk of 50 twice, the second pass starting on a repeat of
    the file before it (loader.py:108-117)."""
    files = sorted(files, key=sequence_sort_key)
    if test_type == "longterm":
        chunks = [files[i:i + 50] for i in range(0, len(files), 50)]
        chunks = sorted(chunks * 2)
        files = [f for c in chunks for f in c]
        for j in range(50, len(files), 100):
            files[j] = files[j - 1]
    return files


def memory_reset_flag(test_type: str, file: str, frame_index: int) -> bool:
    """loader.py:289-293."""
    if test_type in ("default", "longterm"):
        return int(file.split("_")[-1].split(".")[0]) == 0 and frame_index == 0
    if test_type == "episodic":
        return frame_index == 0
    raise ValueError(f"unknown TEST_TYPE {test_type!r}")


class EpisodeDataset:
    """Iteration contract of SMNetDetectionLoader (loader.py:58-308) for the memory path: item = one episode = list of
    <= ``max_sequence_length`` frame dicts with the keys the meta-architecture consumes (train_mp3d.py:474-496):
    ``sequence_name, proj_indices (H,W,1) int32, memory_reset, memory_features, observations`` (+ ``image`` and ``depth``
    when the sensor store holds them).  Detection ground truth and JPEG decoding stay with the detector's data stack."""

    def __init__(self, data_path: str, test_type: str = "default", memory_type: str = "implicit_memory",
                 semmap_path: Optional[str] = None, max_sequence_length: int = 20):
        self.memory_path = os.path.join(data_path, "memory_data")
        self.data_path = os.path.join(data_path, "sensor_data")
        self.test_type, self.memory_type, self.semmap_path = test_type, memory_type, semmap_path
        self.max_sequence_length = max_sequence_length
        if not os.path.isdir(self.memory_path):
            raise StoreError(f"{self.memory_path} does not exist")
        self.files = order_files(os.listdir(self.memory_path), test_type)
        if not self.files:
            raise StoreError(f"{self.memory_path} is empty")          # loader.py:165 asserts the same

    def __len__(self) -> int:
        return len(self.files)

    def __getitem__(self, index: int) -> List[dict]:
        file = self.files[index]
        mem = open_store(os.path.join(self.memory_path, file))
        proj = mem["proj_indices"]
        implicit_memory, observations = mem["memory_features"], None
        if self.semmap_path and os.path.exists(self.semmap_path):                       # loader.py:216-223
            _, implicit_memory, observations = load_memory(os.path.join(self.semmap_path, file))
        sensor = None
        for p in _candidates(os.path.join(self.data_path, file)):
            if os.path.isfile(p):
                sensor = open_store(p)
                break
        frames = []
        for i in range(min(self.max_sequence_length, proj.shape[0])):
            fr = {"sequence_name": file, "proj_indices": proj[i], "memory_reset": memory_reset_flag(self.test_type, file, i)}
            if self.memory_type in ("explicit_map", "implicit_memory"):                  # loader.py:298-303
                fr["memory_features"], fr["observations"] = implicit_memory, observations
            else:
                fr["memory_features"], fr["observations"] = mem["memory_features"], None
            if sensor is not None:
                for k_src, k_dst in (("rgb", "image"), ("depth", "depth")):
                    if k_src in sensor:
                        fr[k_dst] = sensor[k_src][i]
            frames.append(fr)
        return frames

    def __iter__(self) -> Iterator[List[dict]]:
        return (self[i] for i in range(len(self)))
