"""The checkpoint file of a Model (Model.save, load_model).

One file holds two pickles: a small header (a magic string, the format version and the C-ABI version of the
library that wrote it), then the payload (the model's host state and every species' downloaded device state,
with no device handle).  The header is read and checked before the payload is unpickled, so a checkpoint of
another format or library version is refused with a clear error.  Unpickling runs code the file names: load only
checkpoints you trust.  Neither reading nor writing needs the CUDA library.
"""
import os
import pickle

MAGIC = 'geonomics_b200 checkpoint'
FORMAT_VERSION = 1


class CheckpointError(ValueError):
    """A file that is not a checkpoint this build can resume."""


def write(path, payload, abi_version):
    """Write `payload` to `path` atomically: a crash while writing leaves any earlier file at `path` whole."""
    header = dict(magic=MAGIC, format=FORMAT_VERSION, abi=int(abi_version))
    tmp = '%s.tmp%d' % (path, os.getpid())
    try:
        with open(tmp, 'wb') as f:
            pickle.dump(header, f, protocol=pickle.HIGHEST_PROTOCOL)
            pickle.dump(payload, f, protocol=pickle.HIGHEST_PROTOCOL)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)


def read(path, abi_version):
    """The payload of the checkpoint at `path`, after its header is checked against FORMAT_VERSION and the
    C-ABI version `abi_version` of the library that is to resume it."""
    with open(path, 'rb') as f:
        try:
            header = pickle.load(f)
        except Exception as e:
            raise CheckpointError('%s is not a geonomics_b200 checkpoint (%s)' % (path, e))
        if not isinstance(header, dict) or header.get('magic') != MAGIC:
            raise CheckpointError('%s is not a geonomics_b200 checkpoint' % path)
        if header.get('format') != FORMAT_VERSION:
            raise CheckpointError('%s has checkpoint format %r; this build reads format %d only'
                                  % (path, header.get('format'), FORMAT_VERSION))
        if header.get('abi') != int(abi_version):
            raise CheckpointError('%s was written by libgnxb200 C-ABI version %r; this build has version %d'
                                  % (path, header.get('abi'), int(abi_version)))
        return pickle.load(f)
