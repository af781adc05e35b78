"""Frame-range sharding of one clip across the GPUs of a box, plus in-order publishing.

Frames are independent (process_frame is a pure function of one (rgb, depth, params) triple,
reference: helper/stereo_core.py:225-311; the driver treats frames idempotently,
sbs_generator.py:178-185), so sharding needs no collective: every rank takes its own frames and
only a barrier closes the clip.

Constraint inherited from the orchestrator (SURVEY.md 8(e)): progress and "done" are inferred from
the MAX sbs_*.png number (helper/workflow_metrics.py:208-227) and the chunker needs gap-free
ranges (chunk_generator.py:140-178).  Two measures keep that true with several writers:
  * block-cyclic assignment (small blocks dealt round-robin) so that all ranks advance through
    the clip together instead of one rank racing ahead in the last block;
  * `InOrderPublisher`: workers write `sbs_N.png` under a hidden temporary name and the publisher
    renames files into place strictly in frame order, so a visible sbs_N.png implies that every
    pending frame before it is visible too.
"""
from __future__ import annotations

import os
import threading
import time
from typing import Callable, List, Optional, Sequence, Tuple

__all__ = ['contiguous_ranges', 'block_cyclic', 'shard_items', 'consecutive_chunks', 'DelayedFree', 'InOrderPublisher',
           'RawFrameSink', 'dist_env', 'barrier', 'all_reduce_max']


def contiguous_ranges(n: int, world: int) -> List[Tuple[int, int]]:
    """GPU g of G gets items [g*ceil(n/G), (g+1)*ceil(n/G)) (SURVEY 8(e) 'Partitioning')."""
    if world < 1:
        raise ValueError('world must be >= 1')
    per = -(-n // world) if n else 0
    return [(min(g * per, n), min((g + 1) * per, n)) for g in range(world)]


def block_cyclic(n: int, world: int, rank: int, block: int = 16) -> List[int]:
    """Indices of rank `rank`: blocks of `block` consecutive items dealt round-robin."""
    if not (0 <= rank < world):
        raise ValueError('rank out of range')
    out: List[int] = []
    for b0 in range(rank * block, n, world * block):
        out.extend(range(b0, min(b0 + block, n)))
    return out


def shard_items(items: Sequence, world: int, rank: int, block: int = 16, mode: str = 'block_cyclic') -> list:
    if mode == 'contiguous':
        a, b = contiguous_ranges(len(items), world)[rank]
        return list(items[a:b])
    return [items[i] for i in block_cyclic(len(items), world, rank, block)]


def consecutive_chunks(items: Sequence, group: int, number: Callable = lambda it: int(it[2])) -> list:
    """`items` cut into chunks of at most `group` consecutive clip frames: a chunk never spans a gap in the frame
    numbers, so it never straddles a shard block or frames that a resumed run skips."""
    chunks: list = []
    run: list = []
    for it in items:
        if run and (number(it) != number(run[-1]) + 1 or len(run) == group):
            chunks.append(run)
            run = []
        run.append(it)
    if run:
        chunks.append(run)
    return chunks


class DelayedFree:
    """Free-space deletion with temporal filtering: the maps of frame g are read by every frame within `radius` of it,
    so its inputs go only once every clip frame in [g - radius, g + radius] has its output (published now, or `done`
    before this run).  Publication is in order, so in a clip without skipped frames this is: once frame g + radius is
    published.  A resumed run then still finds every map it needs.  `free(number)` deletes the inputs of one frame."""

    def __init__(self, clip_numbers, done_numbers, radius: int, free: Callable[[int], None]):
        self._clip = set(int(n) for n in clip_numbers)
        self._done = set(int(n) for n in done_numbers)
        self._pending: set = set()
        self._k = int(radius)
        self._free = free
        self._lock = threading.Lock()

    def published(self, number: int) -> None:
        number = int(number)
        with self._lock:
            self._done.add(number)
            self._pending.add(number)
            ready = [g for g in range(number - self._k, number + self._k + 1) if g in self._pending and
                     all(x not in self._clip or x in self._done for x in range(g - self._k, g + self._k + 1))]
            for g in ready:
                self._pending.discard(g)
        for g in ready:
            self._free(g)


class InOrderPublisher:
    """Renames finished outputs into place strictly in the order of `final_paths`.

    Workers (any rank / process) call `staged_path(final)` to know where to write and
    `mark_ready(final)` when the file is complete (an atomic rename to `<final>.ready`); a frame that cannot
    be produced (unreadable input, failed save) is reported with `mark_skipped(final)` so that the frames
    after it are not held back (the reference logs such a frame and carries on, sbs_generator.py:229-230).
    One publisher (rank 0) runs `publish_available()` / `run()`, which moves `.ready` files to their final
    names in order, steps over skipped ones and stops at the first frame that is neither.
    `on_published(index)` runs after the final rename of a frame (the place to delete its inputs: not before
    the output exists under its real name).  Safe to call from several threads.
    """

    def __init__(self, final_paths: Sequence[str], on_published: Optional[Callable[[int], None]] = None):
        self.final_paths = [str(p) for p in final_paths]
        self._next = 0
        self._stop = threading.Event()
        self._lock = threading.Lock()
        self._on_published = on_published
        self.skipped: List[str] = []

    @staticmethod
    def staged_path(final: str) -> str:
        d, b = os.path.split(str(final))
        return os.path.join(d, '.' + b + '.part')

    @staticmethod
    def ready_path(final: str) -> str:
        return str(final) + '.ready'

    @staticmethod
    def skip_path(final: str) -> str:
        d, b = os.path.split(str(final))
        return os.path.join(d, '.' + b + '.skip')

    @classmethod
    def mark_ready(cls, final: str) -> None:
        os.replace(cls.staged_path(final), cls.ready_path(final))

    @classmethod
    def mark_skipped(cls, final: str) -> None:
        with open(cls.skip_path(final), 'w'):
            pass

    def publish_available(self) -> int:
        n = 0
        with self._lock:
            while self._next < len(self.final_paths):
                final = self.final_paths[self._next]
                ready, skip = self.ready_path(final), self.skip_path(final)
                published = False
                if os.path.exists(ready):
                    try:
                        os.replace(ready, final)
                        published = True
                    except FileNotFoundError:      # another publisher (process) was faster
                        pass
                elif os.path.exists(skip):
                    try:
                        os.remove(skip)
                    except FileNotFoundError:
                        pass
                    self.skipped.append(final)
                elif not os.path.exists(final):
                    break
                if published and self._on_published is not None:
                    self._on_published(self._next)
                self._next += 1
                n += 1
        return n

    @property
    def published(self) -> int:
        return self._next

    def done(self) -> bool:
        return self._next >= len(self.final_paths)

    def run(self, poll_s: float = 0.05, on_progress: Optional[Callable[[int], None]] = None, timeout_s: Optional[float] = None,
            final: bool = False) -> bool:
        """Publish until everything is visible, stop() is called (ignored when `final`: the last drain after the
        workers have finished) or the timeout passes.  True if every frame is published or skipped."""
        t0 = time.time()
        while not self.done() and (final or not self._stop.is_set()):
            if self.publish_available() and on_progress:
                on_progress(self._next)
            if self.done():
                break
            if timeout_s is not None and time.time() - t0 > timeout_s:
                return False
            time.sleep(poll_s)
        return self.done()

    def stop(self) -> None:
        self._stop.set()


class RawFrameSink:
    """In-order hand-off of packed SBS frames to an encoder, skipping the `sbs_*.png` intermediate
    (SURVEY.md 8(f) rank 2; the consumer today is chunk_generator.py:241-254, which re-decodes the PNGs
    and feeds libx265).

    Worker threads `put(index, frame)` finished frames in any order; one writer thread emits them strictly
    in clip order as raw `rgb24` into a single byte stream (a file, a FIFO an encoder reads from, or '-'
    for stdout), e.g.

        ffmpeg -f rawvideo -pix_fmt rgb24 -s 3840x1080 -r 24 -i sbs.rgb -c:v libx265 ... out.mkv

    A JSON side-car (`<path>.json`, not written for '-') records the geometry and the frame numbers.
    `put` blocks while a frame is more than `max_ahead` positions ahead of the write cursor, so memory
    stays bounded when one GPU runs ahead of another.

    `pixfmt` (stereo_core.PIXFMTS) is the format of the frames the library hands over: with 'yuv420p' or
    'yuv420p10le' a frame is the I420 planes of a `width` x `height` picture as one [height * 3 // 2, width] array
    (uint8 / uint16), limited range, centre-sited chroma, in `matrix`.  The encoder then reads its input format
    directly, and the side-car's `ffmpeg_input` tags the stream's colour description, e.g.

        ffmpeg -f rawvideo -pix_fmt yuv420p10le -s 3840x1080 -color_range tv -colorspace bt709 ... -i sbs.yuv ...
    """

    # ffmpeg's names of the colour description of each YUV matrix (-colorspace, -color_primaries, -color_trc)
    _FFMPEG_COLOUR = {'bt709': 'bt709', 'bt601': 'smpte170m'}

    def __init__(self, path: str, n_frames: int, height: int, width: int, max_ahead: int = 256, frame_numbers=None,
                 pixfmt: str = 'rgb24', matrix: str = 'bt709'):
        import json
        import numpy as np
        from .stereo_core import matrix_code, output_dtype
        self.path, self.n, self.h, self.w = str(path), int(n_frames), int(height), int(width)
        self.dtype = output_dtype(pixfmt)             # ValueError for an unknown format
        matrix_code(matrix)
        if pixfmt != 'rgb24' and (self.h % 2 or self.w % 2):
            raise ValueError(f'{pixfmt} needs an even frame size, got {self.w}x{self.h}')
        self.pixfmt, self.matrix = pixfmt, matrix
        self.shape = (self.h, self.w, 3) if pixfmt == 'rgb24' else (self.h * 3 // 2, self.w)
        self.bytes_per_frame = int(np.prod(self.shape)) * self.dtype.itemsize
        self.max_ahead = int(max_ahead)
        self._pending = {}
        self._next = 0
        self._cv = threading.Condition()
        self._error: Optional[BaseException] = None
        self._closed = False
        if self.path == '-':
            import sys
            self._f = sys.__stdout__.buffer     # the driver moves its own messages to stderr in this mode
        else:
            self._f = open(self.path, 'wb')
            meta = {'pix_fmt': pixfmt, 'width': self.w, 'height': self.h, 'frames': self.n,
                    'bytes_per_frame': self.bytes_per_frame,
                    'frame_numbers': list(frame_numbers) if frame_numbers is not None else None,
                    'ffmpeg_input': f'-f rawvideo -pix_fmt rgb24 -s {self.w}x{self.h} -i {self.path}'}
            if pixfmt != 'rgb24':
                c = self._FFMPEG_COLOUR[matrix]
                meta.update(matrix=matrix, range='tv', chroma_location='center',
                            ffmpeg_input=f'-f rawvideo -pix_fmt {pixfmt} -s {self.w}x{self.h} -color_range tv -colorspace {c} '
                                         f'-color_primaries {c} -color_trc {c} -i {self.path}')
            with open(self.path + '.json', 'w') as jf:
                json.dump(meta, jf)
        self._t = threading.Thread(target=self._run, name='raw-sink', daemon=True)
        self._t.start()

    def put(self, index: int, frame) -> None:
        if frame.shape != self.shape or frame.dtype != self.dtype:
            raise ValueError(f'frame {index}: expected {self.dtype} {self.shape}, got {frame.dtype} {frame.shape}')
        with self._cv:
            while index - self._next > self.max_ahead and self._error is None:
                self._cv.wait(0.1)
            if self._error is not None:
                raise RuntimeError(f'raw sink failed: {self._error}')
            self._pending[int(index)] = frame
            self._cv.notify_all()

    def skip(self, index: int) -> None:
        """A frame that could not be produced (load error): keep the stream gap-free with a black frame (in YUV:
        Y 16 / 64, chroma 128 / 512 at 8 / 10 bits)."""
        import numpy as np
        if self.pixfmt == 'rgb24':
            self.put(index, np.zeros(self.shape, np.uint8))
            return
        black = np.empty(self.shape, self.dtype)
        black[:self.h] = 16 if self.pixfmt == 'yuv420p' else 64
        black[self.h:] = 128 if self.pixfmt == 'yuv420p' else 512
        self.put(index, black)

    @property
    def written(self) -> int:
        return self._next

    def _run(self) -> None:
        try:
            while True:
                with self._cv:
                    while self._next not in self._pending:
                        if self._closed or self._next >= self.n:
                            return
                        self._cv.wait(0.1)
                    frame = self._pending.pop(self._next)
                self._f.write(memoryview(frame).cast('B') if frame.flags['C_CONTIGUOUS'] else frame.tobytes())
                with self._cv:
                    self._next += 1
                    self._cv.notify_all()
        except BaseException as e:   # noqa: BLE001  (a broken pipe must reach the producers)
            with self._cv:
                self._error = e
                self._cv.notify_all()

    def close(self, timeout_s: float = 600.0) -> bool:
        """Write out everything that is contiguous with the cursor, then stop.  True if the whole clip was written."""
        with self._cv:
            self._closed = True       # the writer keeps going while the next frame is there and stops at the first gap
            self._cv.notify_all()
        self._t.join(timeout=timeout_s)
        if self.path != '-':
            self._f.close()
        else:
            self._f.flush()
        if self._error is not None:
            raise RuntimeError(f'raw sink failed: {self._error}')
        return self._next >= self.n


# ---- torch.distributed plumbing (NCCL on GPUs, gloo in CPU tests); no data-path collective -------------
def dist_env() -> Tuple[int, int, int]:
    """(rank, world, local_rank) from the torchrun environment (1 process per GPU)."""
    return int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1')), int(os.environ.get('LOCAL_RANK', '0'))


def barrier() -> None:
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.barrier()
    except ImportError:
        pass


def all_reduce_max(value: float, device: str = 'cpu') -> float:
    """max over ranks of a host scalar (used for timing: a multi-GPU number is the slowest rank's)."""
    try:
        import torch
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            t = torch.tensor([value], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0])
    except ImportError:
        pass
    return float(value)
