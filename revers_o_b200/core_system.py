"""Drop-in for the reference's `core_system.SimpleReverso` on the region-similarity hot path.

Same class name, method names, argument meaning, return shapes and status-string error convention as
/root/reference core_system.py:44-757, so that the unmodified `ui.py` keeps working
(`from core_system import SimpleReverso`, ui.py:19-20).  What changes is what runs underneath:

  extract_embeddings / process_image_direct_pe  (core_system.py:320-455)
        -> K1 mask-pool + L2-normalise CUDA kernel (`ops.mask_pool`) / `ops.normalize_rows`
  create_database ingest tail                   (core_system.py:593-625)
        -> `B200VectorDB.recreate_collection` + `upsert` (bf16 rows on the GPU)
  search_similar query head                     (core_system.py:650-666)
        -> `B200VectorDB.search` (K2 scan + exact select + fp32 re-score)

Out of scope and therefore not re-implemented (SURVEY.md §2): the PE encoder and the GroundedSAM detector.  They can be
injected (`encoder(image_tensor) -> [1,N,D] | [1,D]`, `preprocess(pil) -> tensor`, `detector(pil, prompt) -> object with
.mask [n,H,W], .confidence, .class_id, .xyxy`); with the no-argument constructor the UI uses (ui.py:20) they are loaded
LAZILY through the reference's own imports and calls (`setup_device` / `load_pe_model`, core_system.py:156-203;
`init_grounded_sam`, :205-224) the first time an image has to be embedded or detected, and a ❌ status is reported if those
third-party packages are absent; nothing on the similarity path depends on them.

Several GPUs: `SimpleReverso(devices=[0, 1, ...])`, or the environment variable RVO_DEVICES ("0,1,2,3" or "all") for the
no-argument constructor — `create_database` / `load_database` then row-shard the collection over those GPUs inside this one
process and `search_similar` scans all shards (vector_db.py).

`parity_mode`:
  "reference"  every non-empty region gets the normalised GLOBAL embedding, what core_system.py:406-407 computes today
               (SURVEY.md F4); bf16 / fp16 tokens are consumed as they are, fp32 tokens are rounded to bf16 for the pooling
               kernel (values then agree with the reference's to bf16 rounding of the tokens, ~1e-3 relative);
  "pooled"     the reference's stated design (main.py:8-9): patch features averaged under each mask.
"""
from __future__ import annotations

import os
import shutil
import uuid

import numpy as np
import torch

from . import ops
from ._lib import RvoError
from .vector_db import B200VectorDB, models

DB_ROOT = "./simple_reverso_db"          # core_system.py:76,95,471
COLLECTION_PREFIX = "simple_reverso_"    # core_system.py:101,597
MAX_REGIONS = 50                         # core_system.py:363
UPSERT_BATCH = 100                       # core_system.py:612


def binarize_mask(mask: np.ndarray) -> np.ndarray:
    """core_system.py:398-400."""
    m = np.asarray(mask)
    if m.dtype == bool:
        return m.astype(np.uint8)
    if np.issubdtype(m.dtype, np.floating):
        return (m > 0.5).astype(np.uint8)
    return m.astype(np.uint8)


def mask_to_patch_grid(mask: np.ndarray, grid: int = 24) -> np.ndarray:
    """Image-resolution mask -> binary patch-grid mask [grid*grid] (rule fixed in DESIGN.md §3: a patch
    is in the region when more than half of its pixels are; a non-empty mask never becomes empty)."""
    m = binarize_mask(mask)
    H, W = m.shape
    rb = (np.arange(grid + 1) * H) // grid
    cb = (np.arange(grid + 1) * W) // grid
    r0, c0 = rb[:-1], cb[:-1]
    r1 = np.minimum(np.maximum(rb[1:], r0 + 1), H)
    c1 = np.minimum(np.maximum(cb[1:], c0 + 1), W)
    ii = np.zeros((H + 1, W + 1), dtype=np.int64)
    ii[1:, 1:] = m.astype(np.int64).cumsum(0).cumsum(1)
    s = ii[r1][:, c1] - ii[r0][:, c1] - ii[r1][:, c0] + ii[r0][:, c0]
    area = np.maximum((r1 - r0)[:, None] * (c1 - c0)[None, :], 1)
    frac = s / area
    out = (frac > 0.5).astype(np.uint8)
    if out.sum() == 0 and m.sum() > 0:
        out.flat[int(np.argmax(frac))] = 1
    return out.reshape(-1)


class SimpleReverso:
    """Simplified visual investigation system (B200-native hot path)."""

    def __init__(self, encoder=None, preprocess=None, detector=None, parity_mode: str = "reference",
                 db_root: str = DB_ROOT, device=None, devices=None):
        print("🚀 Initializing Simple Revers-o (B200-native similarity path)...")
        if parity_mode not in ("reference", "pooled"):
            raise ValueError("parity_mode must be 'reference' or 'pooled'")
        self.parity_mode = parity_mode
        self.db_root = db_root
        self.device = torch.device(device) if device is not None else self.setup_device()
        if devices is None and os.environ.get("RVO_DEVICES"):
            spec = os.environ["RVO_DEVICES"].strip().lower()
            devices = list(range(torch.cuda.device_count())) if spec == "all" else [int(x) for x in spec.split(",") if x.strip()]
        self.devices = list(devices) if devices else None      # None: the vector DB lives on self.device only
        self.pe_model, self.preprocess = encoder, preprocess   # None: loaded lazily (load_pe_model) on first use
        self._detector = detector
        self.grounded_sam = None
        self.vector_db = None
        self.current_database = None
        self.detected_regions = []
        self.region_embeddings = None
        self.query_embedding_for_search = None
        self._stop_requested = False
        self._last_processed_file = None
        self._partial_embeddings = []
        self._partial_metadata = []
        print("✅ Simple Revers-o ready!")

    # ---- device / encoder / detector boundary (core_system.py:156-224; third-party, loaded lazily) ---------------
    def setup_device(self):
        """core_system.py:156-167, minus MPS: the similarity path is CUDA (sm_100) only."""
        if torch.cuda.is_available():
            device = torch.device("cuda")
            print(f"🔥 Using CUDA: {device}")
        else:
            device = torch.device("cpu")
            print(f"💻 Using CPU: {device} (embedding only: the vector search needs a B200)")
        return device

    def load_pe_model(self):
        """core_system.py:169-203 through the reference's own imports: PE-Core-L14-336 if available, `.half()` on CUDA
        (mixed precision, :195-196), 336-px transform (:200).  Raises ImportError when perception_models is not installed."""
        import sys
        if "./perception_models" not in sys.path:
            sys.path.append("./perception_models")          # core_system.py:5
        import core.vision_encoder.pe as pe                  # noqa: E402  (third-party, not vendored)
        import core.vision_encoder.transforms as transforms  # noqa: E402
        print("📚 Loading PE-Core-L14-336 (optimal for investigation)...")
        available_configs = pe.CLIP.available_configs()
        target_model = "PE-Core-L14-336"
        name = target_model if target_model in available_configs else available_configs[0]
        try:
            pe_model = pe.CLIP.from_config(name, pretrained=True)
            print(f"✅ Loaded {name}")
        except Exception as e:
            print(f"❌ Failed to load {name}: {e}")
            pe_model = pe.CLIP.from_config(available_configs[0], pretrained=True)
            print(f"🔄 Using fallback: {available_configs[0]}")
        pe_model = pe_model.to(self.device)
        if self.device.type == "cuda":
            pe_model = pe_model.half()
            print("⚡ Mixed precision enabled")
        preprocess = transforms.get_image_transform(336)
        print("🎯 PE model ready - using layer 24 (research optimal)")
        return pe_model, preprocess

    def init_grounded_sam(self, text_prompt):
        """core_system.py:205-224 through the reference's own imports (re-created per call, thresholds 0.35 / 0.25)."""
        from autodistill_grounded_sam import GroundedSAM     # third-party, not vendored
        from autodistill.detection import CaptionOntology
        prompts = [p.strip() for p in text_prompt.split(".") if p.strip()] if text_prompt else []
        if not prompts:
            prompts = ["object"]
        self.grounded_sam = GroundedSAM(ontology=CaptionOntology({p: p for p in prompts}), box_threshold=0.35,
                                        text_threshold=0.25)
        print(f"🎯 GroundedSAM ready with prompts: {prompts}")

    def _detect_with_grounded_sam(self, pil, text_prompt):
        """core_system.py:248-308: temp JPEG round trip, predict, masks to numpy."""
        import tempfile
        self.init_grounded_sam(text_prompt)
        temp_path = os.path.join(tempfile.gettempdir(), f"temp_image_{uuid.uuid4().hex[:8]}.jpg")
        pil.convert("RGB").save(temp_path)
        try:
            det = self.grounded_sam.predict(temp_path)
        finally:
            if os.path.exists(temp_path):
                os.remove(temp_path)
        masks = getattr(det, "mask", None)
        if masks is None:
            masks = getattr(det, "masks", None)
        if isinstance(masks, torch.Tensor):
            masks = masks.detach().cpu().numpy()
        if len(det.xyxy) == 0:
            masks = np.zeros((0, pil.height, pil.width), dtype=np.uint8)
        try:
            from supervision.detection.core import Detections
            return Detections(xyxy=det.xyxy, mask=masks, confidence=det.confidence, class_id=det.class_id)
        except ImportError:
            from types import SimpleNamespace

            class _Det(SimpleNamespace):
                def __len__(self):
                    return len(self.xyxy)
            return _Det(xyxy=det.xyxy, mask=masks, confidence=det.confidence, class_id=det.class_id)

    def _new_client(self, db_path):
        return B200VectorDB(path=db_path, device=self.device if self.device.type == "cuda" else None, devices=self.devices)

    # ---- database housekeeping (core_system.py:74-154) ------------------------------------------
    def list_databases(self):
        if not os.path.exists(self.db_root):
            return []
        return [n for n in os.listdir(self.db_root) if os.path.isdir(os.path.join(self.db_root, n))]

    def load_database(self, database_name):
        if not database_name:
            return "❌ Please provide a database name"
        db_path = f"{self.db_root}/{database_name}"
        if not os.path.exists(db_path):
            return f"❌ Database not found: {database_name}"
        try:
            client = self._new_client(db_path)
            collection_name = f"{COLLECTION_PREFIX}{database_name}"
            names = [c.name for c in client.get_collections().collections]
            if collection_name not in names:
                if database_name in names:  # legacy naming, core_system.py:107-109
                    collection_name = database_name
                else:
                    return f"❌ Collection not found in database: {database_name}"
            self.vector_db = client
            self.current_database = collection_name
            return f"✅ Loaded database: {database_name}"
        except Exception as e:  # status strings, never raise into Gradio
            return f"❌ Error loading database: {str(e)}"

    def delete_database(self, database_name):
        if not database_name:
            return "❌ Please provide a database name"
        db_path = f"{self.db_root}/{database_name}"
        if not os.path.exists(db_path):
            return f"❌ Database not found: {database_name}"
        try:
            if self.current_database in (f"{COLLECTION_PREFIX}{database_name}", database_name):
                self.vector_db = None
                self.current_database = None
            shutil.rmtree(db_path)
            return f"✅ Deleted database: {database_name}"
        except Exception as e:
            return f"❌ Error deleting database: {str(e)}"

    def unlock_database(self, database_name):
        """core_system.py:137-154."""
        if not database_name:
            return "❌ Please provide a database name"
        db_path = f"{self.db_root}/{database_name}"
        if not os.path.exists(db_path):
            return f"❌ Database not found: {database_name}"
        lock_file = os.path.join(db_path, ".lock")
        if os.path.exists(lock_file):
            try:
                os.remove(lock_file)
                return f"✅ Removed lock file from database: {database_name}"
            except Exception as e:
                return f"❌ Error removing lock file: {str(e)}"
        return f"ℹ️ No lock file found for database: {database_name}"

    # ---- detection (third-party; injected) -------------------------------------------------------
    def detect_regions(self, image, text_prompt=None):
        """core_system.py:237-318.  Returns the number of regions; the detector only PRODUCES masks.  Like the reference it
        falls back to the generic prompt "object" and clears the previous detections / embeddings first (:239-246)."""
        if text_prompt is None:
            text_prompt = "object"
        print(f"🔍 Detecting regions with prompt: '{text_prompt}'")
        self.detected_regions = []
        self.region_embeddings = None
        self.query_embedding_for_search = None
        try:
            pil = self._to_pil(image)
            if self._detector is None:
                try:
                    self.detected_regions = self._detect_with_grounded_sam(pil, text_prompt)
                except ImportError as e:
                    return 0 if self._fail(f"GroundedSAM detector not available in this environment ({e})") else 0
            else:
                self.detected_regions = self._detector(pil, text_prompt)
            n = len(self.detected_regions) if self.detected_regions is not None else 0
            print(f"✅ Found {n} regions")
            return n
        except Exception as e:
            print(f"❌ Detection error: {e}")
            self.detected_regions = []
            return 0

    # ---- embedding half --------------------------------------------------------------------------
    def _encode(self, image):
        if self.pe_model is None or self.preprocess is None:
            try:        # the no-argument constructor of ui.py:20: load the reference's own encoder on first use
                self.pe_model, self.preprocess = self.load_pe_model()
            except ImportError as e:
                raise RvoError("PE encoder not available: perception_models is not installed "
                               f"({e}); pass encoder= and preprocess=") from None
        pil = self._to_pil(image)
        x = self.preprocess(pil.convert("RGB")).unsqueeze(0).to(self.device)
        with torch.no_grad():
            fn = getattr(self.pe_model, "encode_image", self.pe_model)
            return fn(x), pil

    def _global_embedding(self, features: torch.Tensor) -> torch.Tensor:
        """core_system.py:345-353 + :407: tokens [1,N,D] -> mean over N -> L2; pooled [1,D] -> L2.
        Both run in the CUDA library: the token mean is K1 with an all-ones mask."""
        if features.dim() == 3:
            _, N, D = features.shape
            feats = self._k1_features(features[:1])               # bf16 / fp16 as they are; fp32 rounded to bf16
            ones = torch.ones((1, 1, N), dtype=torch.uint8, device=feats.device)
            out, _, _, _ = ops.mask_pool(feats, ones)
            return out[0]
        if features.dim() == 2:
            _, f32 = ops.normalize_rows(features[:1].float().contiguous(), want_f32=True)
            return f32[0]
        raise ValueError(f"Unexpected feature shape: {tuple(features.shape)}")

    @staticmethod
    def _k1_features(tokens: torch.Tensor) -> torch.Tensor:
        """K1 consumes 16-bit features: bf16, or the fp16 a `.half()` encoder emits (core_system.py:195-196), unchanged."""
        if tokens.dtype in (torch.bfloat16, torch.float16):
            return tokens.contiguous()
        return tokens.to(torch.bfloat16).contiguous()

    def extract_embeddings(self, image):
        """core_system.py:320-429.  Returns (list[Tensor[D]] on CPU, list[dict])."""
        if self.detected_regions is None or len(self.detected_regions) == 0:
            print("❌ No regions detected")
            return [], []
        try:
            features, pil = self._encode(image)
        except Exception as e:
            print(f"❌ {e}")
            return [], []
        if features.dim() not in (2, 3):
            print(f"[ERROR] Unexpected feature shape: {features.shape}")
            return [], []
        det = self.detected_regions
        masks = getattr(det, "mask", None)
        n_reg = min(len(det), MAX_REGIONS)
        conf = getattr(det, "confidence", None)
        cls = getattr(det, "class_id", None)
        names = self._class_names()

        keep, metas = [], []
        for i in range(n_reg):
            raw_conf = float(conf[i]) if conf is not None and i < len(conf) else 0.0
            cid = int(cls[i]) if cls is not None and i < len(cls) else -1
            if masks is None or i >= len(masks):
                dc = names[cid] if 0 <= cid < len(names) else "unknown"
                keep.append((i, None))
                metas.append({"region_id": str(uuid.uuid4()), "bbox": [0, 0, pil.width, pil.height], "area_ratio": 1.0,
                              "detection_index": i, "confidence": raw_conf, "detected_class": dc,
                              "mask_status": "missing_or_unavailable"})
                continue
            m = binarize_mask(masks[i])
            if m.sum() == 0:  # core_system.py:402-404: dropped, later regions shift up
                print(f"⚠️ Empty mask for region {i}, skipping")
                continue
            ys, xs = np.where(m)
            dc = names[cid] if 0 <= cid < len(names) else "object"
            keep.append((i, m))
            metas.append({"region_id": str(uuid.uuid4()),
                          "bbox": [int(xs.min()), int(ys.min()), int(xs.max()), int(ys.max())],
                          "area_ratio": float(m.sum() / m.size), "detection_index": i, "confidence": raw_conf,
                          "detected_class": dc, "mask_status": "processed"})

        embeddings = []
        if keep:
            pooled_ok = self.parity_mode == "pooled" and features.dim() == 3
            if pooled_ok:
                embeddings = self._pooled_embeddings(features, [m for _, m in keep])
            else:
                g = self._global_embedding(features).cpu()
                embeddings = [g.clone() for _ in keep]
        self.region_embeddings = embeddings
        print(f"🎯 Extracted {len(embeddings)} region embeddings")
        return embeddings, metas

    def _pooled_embeddings(self, features: torch.Tensor, masks_hw: list):
        """north_star path: patch tokens averaged under each mask (K1).  A leading class token is
        dropped when N is not a perfect square but N-1 is."""
        _, N, D = features.shape
        g = int(round(np.sqrt(N)))
        tokens = features[0]
        if g * g != N:
            g = int(round(np.sqrt(N - 1)))
            if g * g != N - 1:
                raise RvoError(f"cannot map {N} tokens to a square patch grid")
            tokens = tokens[1:]
        P = g * g
        M = len(masks_hw)
        pm = np.ones((1, M, P), dtype=np.uint8)
        for j, m in enumerate(masks_hw):
            if m is not None:
                pm[0, j] = mask_to_patch_grid(m, g)
        feats = self._k1_features(tokens).unsqueeze(0)
        out, counts, src, total = ops.mask_pool(feats, torch.from_numpy(pm).to(feats.device))
        out = out[:M].cpu()  # every mask is non-empty here, so total == M
        return [out[j].clone() for j in range(M)]

    def process_image_direct_pe(self, image):
        """core_system.py:431-455."""
        print("🧠 Processing image directly with PE...")
        features, pil = self._encode(image)
        emb = self._global_embedding(features).cpu()
        self.region_embeddings = [emb]
        meta = {"region_id": str(uuid.uuid4()), "bbox": [0, 0, pil.width, pil.height], "area_ratio": 1.0,
                "detection_index": 0, "confidence": 1.0, "detected_class": "full_image"}
        print("✅ Extracted global image embedding")
        return [emb], [meta]

    def request_stop(self):
        """core_system.py:457-459."""
        self._stop_requested = True

    # ---- ingest ------------------------------------------------------------------------------------
    def create_database(self, folder_path, database_name, text_prompt="person . car . building", use_direct_pe=False,
                        progress_callback=None, resume_from_checkpoint=False, include_subfolders=False):
        """core_system.py:461-648: same signature, defaults, status lines and return text.  The checkpoint feature is dead
        code in the reference (json/datetime never imported, SURVEY.md F6) and is not reproduced: `resume_from_checkpoint`
        is accepted and ignored."""
        status_messages = []

        def log_status(message, progress_value=None):
            print(message)
            status_messages.append(message)
            if progress_callback:
                try:
                    progress_callback(message, progress_value)
                except Exception:
                    pass
            return "\n".join(status_messages)

        try:
            if not os.path.exists(folder_path):
                return log_status(f"❌ Folder not found: {folder_path}")
            if not database_name:
                return log_status("❌ Please provide a database name")
            os.makedirs(self.db_root, exist_ok=True)
            db_path = os.path.join(self.db_root, database_name)
            log_status(f"📁 Creating database '{database_name}' from {folder_path}")
            image_extensions = (".jpg", ".jpeg", ".png", ".bmp", ".tiff", ".webp")
            image_files = []
            if include_subfolders:
                for root, _, fs in os.walk(folder_path):
                    image_files += [os.path.join(root, f) for f in fs if f.lower().endswith(image_extensions)]
            else:
                image_files = [os.path.join(folder_path, f) for f in os.listdir(folder_path) if f.lower().endswith(image_extensions)]
            image_files.sort()                      # the reference keeps os.listdir order (arbitrary); sorted is one such order
            if not image_files:
                return log_status(f"❌ No images found in {folder_path}")
            log_status(f"📊 Found {len(image_files)} images to process", 0.1)
            if include_subfolders:
                log_status("📂 Including images from subfolders")
            log_status(f"🔧 Processing mode: {'Direct PE' if use_direct_pe else 'GroundedSAM + PE'}")
            log_status(f"📂 Database will be stored at: {db_path}")

            os.makedirs(db_path, exist_ok=True)
            client = self._new_client(db_path)          # persists implicitly on every upsert, like QdrantClient(path=...)
            processed = failed = 0
            for i, image_path in enumerate(image_files):
                if self._stop_requested:
                    log_status("🛑 Stop requested. Saving progress...")
                    return "\n".join(status_messages) + "\n\n⏸️ Processing stopped. You can resume later."
                filename = os.path.basename(image_path)
                log_status(f"🔄 Processing {i + 1}/{len(image_files)}: {filename}", 0.1 + (0.7 * (i / len(image_files))))
                try:
                    from PIL import Image
                    image = Image.open(image_path).convert("RGB")
                    if use_direct_pe:
                        embeddings, metadata_list = self.process_image_direct_pe(image)
                        log_status(f"✅ Extracted global embedding for {filename}")
                    else:
                        num_regions = self.detect_regions(image, text_prompt)
                        if num_regions > 0:
                            embeddings, metadata_list = self.extract_embeddings(image)
                            log_status(f"✅ Found {num_regions} regions, extracted {len(embeddings)} embeddings in {filename}")
                        else:
                            log_status(f"⚠️ No regions found in {filename}, skipping")
                            failed += 1
                            continue
                    for meta_item in metadata_list:
                        meta_item["image_source"] = image_path
                        meta_item["filename"] = filename
                        # a new UUID per point; the extraction-time id is kept in the payload (core_system.py:571-574)
                        meta_item["original_region_id"] = meta_item.get("region_id", str(uuid.uuid4()))
                        meta_item["region_id"] = str(uuid.uuid4())
                    self._partial_embeddings.extend(embeddings)
                    self._partial_metadata.extend(metadata_list)
                    processed += 1
                    self._last_processed_file = image_path
                except Exception as e:
                    log_status(f"❌ Error processing {filename}: {str(e)}")
                    failed += 1
                    continue
            if not self._partial_embeddings:
                return log_status("❌ No embeddings extracted from any images")

            vector_dim = self._partial_embeddings[0].shape[0]
            collection_name = f"{COLLECTION_PREFIX}{database_name}"
            try:
                client.recreate_collection(collection_name=collection_name,
                                           vectors_config=models.VectorParams(size=vector_dim, distance=models.Distance.COSINE))
                log_status(f"📦 Recreated collection: {collection_name}", 0.8)
            except Exception as e:
                log_status(f"ℹ️ Note: Collection {collection_name} might already exist or error: {e}")
            points = [models.PointStruct(id=meta["region_id"], vector=emb.cpu().numpy(), payload=meta)
                      for emb, meta in zip(self._partial_embeddings, self._partial_metadata)]
            for j in range(0, len(points), UPSERT_BATCH):
                if self._stop_requested:
                    log_status("🛑 Stop requested during database storage. Progress saved.")
                    return "\n".join(status_messages) + "\n\n⏸️ Processing stopped. You can resume later."
                batch_points = points[j:j + UPSERT_BATCH]
                client.upsert(collection_name=collection_name, points=batch_points)
                log_status(f"💾 Stored batch {j // UPSERT_BATCH + 1}/{(len(points) + UPSERT_BATCH - 1) // UPSERT_BATCH} "
                           f"({len(batch_points)} points)", 0.8 + (0.1 * (j / len(points))))
            self.vector_db = client
            self.current_database = collection_name
            log_status("\n📊 Final Summary:", 0.9)
            log_status(f"✅ Successfully processed: {processed} images")
            if failed > 0:
                log_status(f"⚠️ Failed to process: {failed} images")
            log_status(f"🔍 Total embeddings stored: {len(self._partial_embeddings)}")
            log_status(f"🎯 Database '{database_name}' ready for searching!", 1.0)
        except Exception as e:                      # the UI shows the text; nothing raises into Gradio (ui.py:102-104)
            log_status(f"❌ Error creating database: {e}")
        finally:
            self._stop_requested = False
            self._partial_embeddings = []
            self._partial_metadata = []
        return "\n".join(status_messages)

    # ---- search ------------------------------------------------------------------------------------
    def search_similar(self, similarity_threshold=0.7, max_results=5):
        """core_system.py:650-717.  Returns (status text, list of dict{image, score, filename, bbox})."""
        if not self.region_embeddings:
            return "❌ No query embeddings available. Please detect/process an image first.", []
        if not self.vector_db or not self.current_database:
            return "❌ No database loaded. Please create or load a database first.", []
        print(f"🔍 Searching for similar regions (threshold={similarity_threshold}, max_results={max_results})")
        query_embedding = self.region_embeddings[0]  # first region is the query, core_system.py:657
        try:
            search_results = self.vector_db.search(
                collection_name=self.current_database,
                query_vector=query_embedding.detach().cpu().numpy(),
                limit=max_results,
                score_threshold=similarity_threshold,
            )
        except Exception as e:
            return f"❌ Search error: {e}", []
        if not search_results:
            return f"❌ No similar regions found above threshold {similarity_threshold}", []

        results_text = f"🎯 Found {len(search_results)} similar regions:\n\n"
        items = []
        for i, result in enumerate(search_results):
            payload = result.payload or {}
            filename = payload.get("filename", "Unknown")
            score = result.score
            image_path = payload.get("image_source", "")
            results_text += f"{i + 1}. {filename} (Similarity: {score:.3f})\n"
            results_text += f"   Source: {image_path}\n"
            results_text += f"   📍 Bounding box: {str(payload.get('bbox', '[0,0,0,0]'))}\n\n"
            items.append({"image": self._thumbnail(image_path, score), "score": score, "filename": filename,
                          "bbox": payload.get("bbox")})
        print(f"📊 Processed {len(items)} search results for display.")
        return results_text, items

    def search_similar_batch(self, similarity_threshold=0.7, max_results=5):
        """New (SURVEY.md §8f row 4): search with ALL region embeddings of the query image at once.
        Returns one `search_similar`-shaped hit list per region."""
        if not self.region_embeddings:
            return "❌ No query embeddings available. Please detect/process an image first.", []
        if not self.vector_db or not self.current_database:
            return "❌ No database loaded. Please create or load a database first.", []
        q = torch.stack([e.detach().float().cpu() for e in self.region_embeddings]).numpy()
        ids, scores, counts = self.vector_db.search_batch(self.current_database, q, max_results, similarity_threshold)
        c = self.vector_db._coll(self.current_database)
        out = []
        for r in range(len(q)):
            hits = []
            for i, s in zip(ids[r, :counts[r]], scores[r, :counts[r]]):
                pay = c.payloads[int(i)] or {}
                hits.append({"image": None, "score": float(s), "filename": pay.get("filename", "Unknown"),
                             "bbox": pay.get("bbox")})
            out.append(hits)
        return f"🎯 Searched {len(q)} regions", out

    def find_shared_regions(self, other_database_name, similarity_threshold=0.95, max_results=20):
        """New: which regions of the loaded database also appear in another database — every pair at cosine >=
        similarity_threshold, found by one join on the GPU (`B200VectorDB.join_collections`) instead of one search per stored
        region.  The other database is opened as `load_database` opens one (same devices, same collection naming).  Returns
        (status text, list of dict{score, filename, bbox, other_filename, other_bbox}) for the `max_results` best pairs: score
        descending, ties by the loaded database's row, then the other database's row."""
        if not self.vector_db or not self.current_database:
            return "❌ No database loaded. Please create or load a database first.", []
        if not other_database_name:
            return "❌ Please provide a database name", []
        db_path = f"{self.db_root}/{other_database_name}"
        if not os.path.exists(db_path):
            return f"❌ Database not found: {other_database_name}", []
        if self.vector_db.path and os.path.realpath(self.vector_db.path) == os.path.realpath(db_path):
            return f"❌ {other_database_name} is the loaded database: choose another database to compare with", []
        other = None
        try:
            other = self._new_client(db_path)
            collection_name = f"{COLLECTION_PREFIX}{other_database_name}"
            names = [c.name for c in other.get_collections().collections]
            if collection_name not in names:
                if other_database_name in names:  # legacy naming, as in load_database
                    collection_name = other_database_name
                else:
                    return f"❌ Collection not found in database: {other_database_name}", []
            print(f"🔍 Joining {self.current_database} with {collection_name} (threshold={similarity_threshold})")
            with self.vector_db._read_both(other):
                a, b, pairs, scores = self.vector_db._join_rows(self.current_database, collection_name, similarity_threshold,
                                                               1 << 22, other)
                best = np.lexsort((pairs[:, 1], pairs[:, 0], -scores))[:max(int(max_results), 0)]
                items = []
                for k in best:
                    pa, pb = a.payloads[int(pairs[k, 0])] or {}, b.payloads[int(pairs[k, 1])] or {}
                    items.append({"score": float(scores[k]), "filename": pa.get("filename", "Unknown"), "bbox": pa.get("bbox"),
                                  "other_filename": pb.get("filename", "Unknown"), "other_bbox": pb.get("bbox")})
        except Exception as e:
            return f"❌ Join error: {e}", []
        finally:
            if other is not None:
                other.close()
        if len(pairs) == 0:
            return f"❌ No shared regions found above threshold {similarity_threshold}", []
        results_text = f"🎯 Found {len(pairs)} shared regions with {other_database_name}, showing {len(items)}:\n\n"
        for i, it in enumerate(items):
            results_text += f"{i + 1}. {it['filename']} ↔ {it['other_filename']} (Similarity: {it['score']:.3f})\n"
            results_text += f"   📍 Bounding boxes: {it['bbox']} ↔ {it['other_bbox']}\n\n"
        return results_text, items

    def find_best_matches(self, other_database_name, similarity_threshold=0.0, max_results=20):
        """New: one-to-one correspondences between the loaded database and another one — the pairs of regions that are each
        other's best match (mutual nearest neighbours) at cosine >= similarity_threshold, from two k = 1 joins on the GPU
        (`B200VectorDB.knn_join`, this database against the other and back; `vector_db.mutual_best`).  The other database is
        opened and checked as `find_shared_regions` does.  Returns (status text, list of dict{score, filename, bbox,
        other_filename, other_bbox}) for the `max_results` best pairs: score descending, ties by the loaded database's row,
        then the other database's row."""
        from .vector_db import mutual_best
        if not self.vector_db or not self.current_database:
            return "❌ No database loaded. Please create or load a database first.", []
        if not other_database_name:
            return "❌ Please provide a database name", []
        db_path = f"{self.db_root}/{other_database_name}"
        if not os.path.exists(db_path):
            return f"❌ Database not found: {other_database_name}", []
        if self.vector_db.path and os.path.realpath(self.vector_db.path) == os.path.realpath(db_path):
            return f"❌ {other_database_name} is the loaded database: choose another database to compare with", []
        other = None
        try:
            other = self._new_client(db_path)
            collection_name = f"{COLLECTION_PREFIX}{other_database_name}"
            names = [c.name for c in other.get_collections().collections]
            if collection_name not in names:
                if other_database_name in names:  # legacy naming, as in load_database
                    collection_name = other_database_name
                else:
                    return f"❌ Collection not found in database: {other_database_name}", []
            print(f"🔍 Matching {self.current_database} with {collection_name} (threshold={similarity_threshold})")
            with self.vector_db._read_both(other):
                r_ab, s_ab, c_ab = self.vector_db._knn_rows(self.current_database, 1, similarity_threshold, collection_name, other)
                r_ba, _, c_ba = other._knn_rows(collection_name, 1, similarity_threshold, self.current_database, self.vector_db)
                pairs, scores = mutual_best(r_ab, c_ab, r_ba, c_ba, s_ab)
                a, b = self.vector_db._coll(self.current_database), other._coll(collection_name)
                items = []
                for (i, j), s in zip(pairs[:max(int(max_results), 0)].tolist(), scores.tolist()):
                    pa, pb = a.payloads[int(i)] or {}, b.payloads[int(j)] or {}
                    items.append({"score": float(s), "filename": pa.get("filename", "Unknown"), "bbox": pa.get("bbox"),
                                  "other_filename": pb.get("filename", "Unknown"), "other_bbox": pb.get("bbox")})
        except Exception as e:
            return f"❌ Match error: {e}", []
        finally:
            if other is not None:
                other.close()
        if len(pairs) == 0:
            return f"❌ No mutual best matches found above threshold {similarity_threshold}", []
        results_text = f"🎯 Found {len(pairs)} one-to-one matches with {other_database_name}, showing {len(items)}:\n\n"
        for i, it in enumerate(items):
            results_text += f"{i + 1}. {it['filename']} ↔ {it['other_filename']} (Similarity: {it['score']:.3f})\n"
            results_text += f"   📍 Bounding boxes: {it['bbox']} ↔ {it['other_bbox']}\n\n"
        return results_text, items

    def find_recurring_regions(self, similarity_threshold=0.95, max_groups=20):
        """New: where does an object or scene recur across the loaded database — the groups of regions connected to each other
        at cosine >= similarity_threshold (single linkage), found on the GPU (`B200VectorDB.find_duplicate_groups`) without
        listing every pair.  Returns (status text, list of dict{size, members: [dict{filename, bbox}, ...]}) for the
        `max_groups` largest groups, largest first, members in the database's order."""
        if not self.vector_db or not self.current_database:
            return "❌ No database loaded. Please create or load a database first.", []
        print(f"🔍 Grouping recurring regions of {self.current_database} (threshold={similarity_threshold})")
        try:
            with self.vector_db._lock.read():
                c = self.vector_db._coll(self.current_database)
                groups = self.vector_db._duplicate_group_rows(self.current_database, similarity_threshold, 2)
                items = []
                for g in groups[:max(int(max_groups), 0)]:
                    members = []
                    for r in g:
                        pay = c.payloads[int(r)] or {}
                        members.append({"filename": pay.get("filename", "Unknown"), "bbox": pay.get("bbox")})
                    items.append({"size": len(g), "members": members})
        except Exception as e:
            return f"❌ Grouping error: {e}", []
        if not groups:
            return f"❌ No recurring regions found above threshold {similarity_threshold}", []
        results_text = f"🎯 Found {len(groups)} groups of recurring regions, showing {len(items)}:\n\n"
        for i, it in enumerate(items):
            files = sorted({m["filename"] for m in it["members"]})
            results_text += f"{i + 1}. {it['size']} regions in {len(files)} images: {', '.join(files[:5])}"
            results_text += f" (+{len(files) - 5} more)\n" if len(files) > 5 else "\n"
            results_text += f"   📍 First region: {it['members'][0]['filename']} {it['members'][0]['bbox']}\n\n"
        return results_text, items

    def find_visual_themes(self, n_themes=20, max_themes=20, examples=5):
        """New: what kinds of regions the loaded database holds, and how many of each — spherical k-means of its regions into
        n_themes clusters on the GPU (`B200VectorDB.cluster`; fewer when the database holds fewer regions).  Returns (status
        text, list of dict{size, images: distinct filenames, examples: [dict{filename, bbox, score}]}) for the `max_themes`
        largest themes, largest first; the examples are the `examples` members nearest their theme's centre (highest score,
        ties by the database's order)."""
        if not self.vector_db or not self.current_database:
            return "❌ No database loaded. Please create or load a database first.", []
        print(f"🔍 Finding visual themes of {self.current_database} (n_themes={n_themes})")
        try:
            with self.vector_db._lock.read():
                c = self.vector_db._coll(self.current_database)
                if c.n == 0:
                    return "❌ The database holds no regions", []
                res = self.vector_db._cluster_rows(self.current_database, min(int(n_themes), c.n), 50, 0, None)
                items = []
                for t in range(min(max(int(max_themes), 0), len(res.sizes))):
                    if res.sizes[t] == 0:
                        break
                    rows = np.flatnonzero(res.labels == t)
                    best = rows[np.lexsort((rows, -res.scores[rows].astype(np.float64)))]
                    pays = [c.payloads[int(r)] or {} for r in rows]
                    ex = []
                    for r in best[:max(int(examples), 0)]:
                        pay = c.payloads[int(r)] or {}
                        ex.append({"filename": pay.get("filename", "Unknown"), "bbox": pay.get("bbox"),
                                   "score": float(res.scores[r])})
                    items.append({"size": int(res.sizes[t]), "images": sorted({p.get("filename", "Unknown") for p in pays}),
                                  "examples": ex})
        except Exception as e:
            return f"❌ Clustering error: {e}", []
        results_text = f"🎯 Found {int((res.sizes > 0).sum())} visual themes in {c.n} regions, showing {len(items)}:\n\n"
        for i, it in enumerate(items):
            files = it["images"]
            results_text += f"{i + 1}. {it['size']} regions in {len(files)} images: {', '.join(files[:5])}"
            results_text += f" (+{len(files) - 5} more)\n" if len(files) > 5 else "\n"
            if it["examples"]:
                e = it["examples"][0]
                results_text += f"   📍 Most typical region: {e['filename']} {e['bbox']} (Similarity: {e['score']:.3f})\n\n"
        return results_text, items

    def visualize_detections(self, image, selected_region_index=None):
        """core_system.py:719-757 — rendering, out of scope; returns the image with region boxes drawn."""
        pil = self._to_pil(image).copy()
        det = self.detected_regions
        boxes = getattr(det, "xyxy", None) if det is not None else None
        if boxes is not None:
            from PIL import ImageDraw
            d = ImageDraw.Draw(pil)
            for i, b in enumerate(boxes):
                colour = "yellow" if selected_region_index is not None and i == selected_region_index else "lime"
                d.rectangle([float(b[0]), float(b[1]), float(b[2]), float(b[3])], outline=colour, width=3)
                d.text((float(b[0]) + 4, float(b[1]) + 4), str(i + 1), fill=colour)
        return pil

    # ---- helpers -----------------------------------------------------------------------------------
    @staticmethod
    def _to_pil(image):
        from PIL import Image
        if isinstance(image, np.ndarray):
            return Image.fromarray(image)
        if isinstance(image, str):
            return Image.open(image)
        return image

    def _class_names(self):
        try:
            return list(self.grounded_sam.ontology.classes())
        except Exception:
            return ["object"]

    @staticmethod
    def _fail(msg):
        print(f"❌ {msg}")
        return True

    @staticmethod
    def _thumbnail(image_path, score):
        if not image_path or not os.path.exists(image_path):
            return None
        try:
            from PIL import Image, ImageDraw
            img = Image.open(image_path).convert("RGB")
            d = ImageDraw.Draw(img)
            text = f"Score: {score:.3f}"
            box = d.textbbox((5, 5), text)
            d.rectangle([box[0] - 2, box[1] - 2, box[2] + 2, box[3] + 2], fill="black")
            d.text((5, 5), text, fill="white")
            img.thumbnail((400, 400))
            return img
        except Exception as e:
            print(f"❌ Error loading/processing image {image_path}: {e}")
            return None
