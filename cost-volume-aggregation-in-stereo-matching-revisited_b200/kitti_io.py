"""Image side of the reference's inference driver (SURVEY 8f rank 4): load + normalise a stereo pair, fit it to the
network's input size, crop the prediction back, write the KITTI 16-bit disparity PNG.  Host-only (numpy / PIL); the
only device work is the model call itself.

Mirrors, function by function:
  load_pair            my_img.py:47-71   per-image, per-channel (x - mean) / std of the 8-bit RGB values
  fit_to_crop          my_img.py:73-89   smaller images: zero-padded at the TOP and RIGHT into crop_h x crop_w;
                                         larger: rows cropped around the centre, columns from 0
  pad_to_multiple      main_dca.py:153-166  top / right zero padding to multiples of 16
  fit_gt_to_crop, pad_gt_to_multiple       the same two framings for a ground-truth disparity map (padding 0 = no GT)
  crop_prediction      my_img.py:105-108, main_dca.py:171-174
  save_disparity_png   my_img.py:110     uint16(disp * 256), the KITTI submission format
  predict_files        my_img.py:91-110
"""
import numpy as np
import torch


def _normalised(img):
    """uint8 [H,W,>=3] -> float32 [3,H,W], each channel standardised by ITS OWN mean/std (population std, np.std)."""
    a = np.asarray(img)
    if a.ndim != 3 or a.shape[2] < 3:
        raise ValueError("expected an RGB image [H, W, 3]")
    out = np.empty((3, a.shape[0], a.shape[1]), np.float32)
    for c in range(3):
        ch = a[:, :, c]
        out[c] = (ch - np.mean(ch)) / np.std(ch)
    return out


def load_pair(left, right):
    """Two file names (or PIL images / uint8 arrays) -> float32 [6,H,W]: left RGB then right RGB, standardised."""
    from PIL import Image
    imgs = [Image.open(x) if isinstance(x, (str, bytes)) or hasattr(x, "__fspath__") else x for x in (left, right)]
    l, r = _normalised(imgs[0]), _normalised(imgs[1])
    if l.shape != r.shape:
        raise ValueError(f"left {l.shape[1:]} and right {r.shape[1:]} images differ in size")
    return np.concatenate([l, r], axis=0)


def fit_to_crop(pair, crop_height=384, crop_width=1248):
    """float32 [6,h,w] -> (left [1,3,crop_h,crop_w], right, h, w) as torch tensors."""
    _, h, w = pair.shape
    if h <= crop_height and w <= crop_width:
        fitted = np.zeros((6, crop_height, crop_width), np.float32)
        fitted[:, crop_height - h:, :w] = pair
    else:
        start_y = int((h - crop_height) / 2)
        fitted = pair[:, start_y:start_y + crop_height, :crop_width]
    fitted = np.ascontiguousarray(fitted, dtype=np.float32)
    return torch.from_numpy(fitted[None, 0:3].copy()), torch.from_numpy(fitted[None, 3:6].copy()), h, w


def pad_to_multiple(img, multiple=16):
    """[B,C,H,W] -> (zero-padded at the top and right to multiples of `multiple`, top_pad, right_pad)."""
    H, W = img.shape[2], img.shape[3]
    top = (-H) % multiple
    right = (-W) % multiple
    return torch.nn.functional.pad(img, (0, right, top, 0)), top, right


def fit_gt_to_crop(gt, crop_height=384, crop_width=1248):
    """Ground truth [h,w] -> float32 [crop_h, crop_w] framed exactly as `fit_to_crop` frames the images, so GT pixel
    (y, x) sits under prediction pixel (y, x); the padding is 0 (= no ground truth)."""
    h, w = gt.shape
    if h <= crop_height and w <= crop_width:
        fitted = np.zeros((crop_height, crop_width), np.float32)
        fitted[crop_height - h:, :w] = gt
        return fitted
    start_y = int((h - crop_height) / 2)
    return np.ascontiguousarray(gt[start_y:start_y + crop_height, :crop_width], dtype=np.float32)


def pad_gt_to_multiple(gt, multiple=16):
    """Ground truth [H,W] -> (float32 zero-padded at the top and right like `pad_to_multiple`, top_pad, right_pad)."""
    H, W = gt.shape
    top, right = (-H) % multiple, (-W) % multiple
    return np.pad(np.asarray(gt, np.float32), ((top, 0), (0, right))), top, right


def crop_prediction(disp, h, w, crop_height=384, crop_width=1248):
    """Undo fit_to_crop on a [crop_h, crop_w] disparity map (no-op for images that were cropped, as in the reference)."""
    if h <= crop_height and w <= crop_width:
        return disp[crop_height - h:crop_height, 0:w]
    return disp


def save_disparity_png(path, disp):
    """KITTI format: 16-bit grayscale PNG of disp * 256 (truncated like numpy's astype('uint16'))."""
    from PIL import Image
    a = (np.asarray(disp, dtype=np.float32) * 256.0).astype("uint16")
    Image.fromarray(a).save(path, format="PNG")       # uint16 arrays map to PIL mode I;16
    return a


def predict_files(model, leftname, rightname, savename=None, crop_height=384, crop_width=1248):
    """my_img.py's `my()`: files in, disparity map [h,w] float32 out (and the PNG written when `savename` is given)."""
    left, right, h, w = fit_to_crop(load_pair(leftname, rightname), crop_height, crop_width)
    dev = next(model.parameters()).device
    model.eval()
    with torch.no_grad():
        out = model(left.to(dev), right.to(dev))
    pred = out[0] if isinstance(out, (tuple, list)) else out      # this repo's GwcNet returns (pred4, prob_volume2)
    disp = crop_prediction(pred.squeeze().detach().float().cpu().numpy(), h, w, crop_height, crop_width)
    if savename is not None:
        save_disparity_png(savename, disp)
    return disp


class ImagePipeline:
    """The loop of my_img.py (`main()` :112-125 calling `my()` :91-110 once per pair, everything serial: decode,
    `.cuda()`, forward, `.cpu()`, PNG write) as a batched pinned-memory pipeline:

      loader threads   decode + standardise + fit (`load_pair`, `fit_to_crop`) the NEXT pairs while the device works
      slot ring        `depth` pinned host input buffers [6, crop_h, crop_w] and pinned output buffers [crop_h, crop_w];
                       H2D of pair i+1 on a copy stream overlaps the kernels of pair i, D2H is asynchronous too
      writer thread    waits for a slot's D2H event, crops the prediction back and writes the KITTI 16-bit PNG

    Results are identical to `predict_files` pair by pair (same functions, same order of operations).  With a CPU model
    (tests) the same code runs without pinned memory and streams."""

    def __init__(self, model, crop_height=384, crop_width=1248, depth=3, workers=2):
        self.model = model
        self.ch, self.cw, self.depth, self.workers = crop_height, crop_width, max(2, depth), max(1, workers)
        try:
            self.dev = next(model.parameters()).device
        except (StopIteration, AttributeError):
            self.dev = torch.device("cpu")
        self.cuda = self.dev.type == "cuda"
        mk = (lambda *s: torch.empty(s, dtype=torch.float32).pin_memory()) if self.cuda else \
            (lambda *s: torch.empty(s, dtype=torch.float32))
        self.in_host = [mk(6, crop_height, crop_width) for _ in range(self.depth)]
        self.out_host = [mk(crop_height, crop_width) for _ in range(self.depth)]
        self.in_dev = [torch.empty((6, crop_height, crop_width), dtype=torch.float32, device=self.dev)
                       for _ in range(self.depth)] if self.cuda else self.in_host
        if self.cuda:
            self.copy_stream = torch.cuda.Stream(device=self.dev)
            self.compute_stream = torch.cuda.Stream(device=self.dev)
            self.h2d = [torch.cuda.Event() for _ in range(self.depth)]
            self.done = [torch.cuda.Event() for _ in range(self.depth)]
            self.free = [torch.cuda.Event() for _ in range(self.depth)]

    def _load(self, left, right):
        pair = load_pair(left, right)
        _, h, w = pair.shape
        if h <= self.ch and w <= self.cw:
            fitted = np.zeros((6, self.ch, self.cw), np.float32)
            fitted[:, self.ch - h:, :w] = pair
        else:
            start_y = int((h - self.ch) / 2)
            fitted = np.ascontiguousarray(pair[:, start_y:start_y + self.ch, :self.cw], dtype=np.float32)
        return fitted, h, w

    def _load_framed(self, left, right, mode):
        """Decode, standardise and frame a pair, keeping the left image under the window: mode "fit" (fit_to_crop) or
        "pad16" (pad_to_multiple(16)) -> (fitted float32 [6,Hn,Wn], left uint8 RGB [h,w,3] of the window (a view of
        the decoded image), window, image height, image width).  window = (y0, x0, h, w, v_origin) selects the image part of a network-frame map
        (geometry.reproject, wls.wls_filter)."""
        from PIL import Image
        imgs = [np.asarray(Image.open(x) if isinstance(x, (str, bytes)) or hasattr(x, "__fspath__") else x)
                for x in (left, right)]
        if mode == "fit":
            fitted, h, w = self._load(imgs[0], imgs[1])
            if h <= self.ch and w <= self.cw:
                window = (self.ch - h, 0, h, w, 0)
                rgb = imgs[0][:, :, :3]
            else:
                top = int((h - self.ch) / 2)
                window = (0, 0, self.ch, self.cw, top)
                rgb = imgs[0][top:top + self.ch, :self.cw, :3]
            return fitted, rgb, window, h, w
        pair = load_pair(imgs[0], imgs[1])
        _, h, w = pair.shape
        fitted, top, _ = pad_to_multiple(torch.from_numpy(pair)[None], 16)
        return fitted[0].numpy(), imgs[0][:, :, :3], (top, 0, h, w, 0), h, w

    def _forward(self, slot):
        x = self.in_dev[slot]
        out = self.model(x[None, 0:3], x[None, 3:6])
        pred = out[0] if isinstance(out, (tuple, list)) else out
        return pred.reshape(self.ch, self.cw).float()

    def run(self, triples):
        """triples: iterable of (leftname, rightname, savename or None).  Returns the list of cropped disparity maps
        (float32 numpy [h, w]) in input order; PNGs are written by the writer thread as results arrive."""
        import queue
        import threading
        from concurrent.futures import ThreadPoolExecutor
        triples = list(triples)
        results = [None] * len(triples)
        slot_sem = threading.Semaphore(self.depth)          # a slot is reusable once the writer has consumed its output
        q = queue.Queue()
        err = []

        def writer():
            while True:
                item = q.get()
                if item is None:
                    return
                i, slot, h, w, savename = item
                try:
                    if self.cuda:
                        self.done[slot].synchronize()
                    disp = crop_prediction(self.out_host[slot].numpy(), h, w, self.ch, self.cw).copy()
                    if savename is not None:
                        save_disparity_png(savename, disp)
                    results[i] = disp
                except Exception as e:          # surfaced by run()
                    err.append(e)
                finally:
                    slot_sem.release()

        wt = threading.Thread(target=writer, daemon=True)
        wt.start()
        was_training = getattr(self.model, "training", False)
        if hasattr(self.model, "eval"):
            self.model.eval()
        try:
            with ThreadPoolExecutor(self.workers) as pool, torch.no_grad():
                futs = [pool.submit(self._load, l, r) for l, r, _ in triples]
                for i, (fut, (_, _, savename)) in enumerate(zip(futs, triples)):
                    fitted, h, w = fut.result()
                    slot_sem.acquire()
                    slot = i % self.depth
                    np.copyto(self.in_host[slot].numpy(), fitted)
                    if self.cuda:
                        with torch.cuda.stream(self.copy_stream):
                            if i >= self.depth:
                                self.copy_stream.wait_event(self.free[slot])     # kernels of the slot's previous pair
                            self.in_dev[slot].copy_(self.in_host[slot], non_blocking=True)
                            self.h2d[slot].record(self.copy_stream)
                        with torch.cuda.stream(self.compute_stream):
                            self.compute_stream.wait_event(self.h2d[slot])
                            pred = self._forward(slot)
                            self.free[slot].record(self.compute_stream)
                            self.out_host[slot].copy_(pred, non_blocking=True)
                            self.done[slot].record(self.compute_stream)
                    else:
                        self.out_host[slot].copy_(self._forward(slot))
                    q.put((i, slot, h, w, savename))
        finally:
            q.put(None)
            wt.join()
            if was_training and hasattr(self.model, "train"):
                self.model.train()
        if err:
            raise err[0]
        return results
