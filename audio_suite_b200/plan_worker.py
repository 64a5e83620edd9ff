"""Planning worker process: `python -m audio_suite_b200.plan_worker`.

Reads length-prefixed pickles of parameter-dict chunks on stdin, answers with length-prefixed pickles of
packed job tables (tables.pack_chunk).  Pure host work (numpy Generators, Python rounding): it never
touches CUDA, and because it is a fresh interpreter started with subprocess it is safe next to an
initialised CUDA context and independent of how the parent's __main__ was started."""
import pickle
import struct
import sys


def main():
    from audio_suite_b200 import plan as P, tables as T
    inp, out = sys.stdin.buffer, sys.stdout.buffer
    while True:
        head = inp.read(8)
        if len(head) < 8:
            return
        (size,) = struct.unpack("<Q", head)
        chunk = pickle.loads(inp.read(size))
        try:
            reply = ("ok", T.pack_chunk([P.plan_render(p) for p in chunk]))
        except BaseException as e:                     # the parent re-raises
            reply = ("err", e)
        blob = pickle.dumps(reply, protocol=pickle.HIGHEST_PROTOCOL)
        out.write(struct.pack("<Q", len(blob)))
        out.write(blob)
        out.flush()


if __name__ == "__main__":
    main()
