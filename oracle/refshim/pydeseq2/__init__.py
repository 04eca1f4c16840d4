"""Import shim (TEST INFRASTRUCTURE).

Makes the reference package importable without installing it, from the byte-compiled copy ``build()`` leaves in
``oracle/_ref/pydeseq2`` (oracle/build_ref.py): the real ``pydeseq2/__init__.py`` calls
``importlib.metadata.version("pydeseq2")``, which fails for an un-installed tree, so this module stands in for it.
Only used by ``oracle/make_golden.py`` and the drop-in tests; nothing on the product path imports it.
"""
import os as _os

__path__ = [_os.path.join(_os.path.dirname(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__)))), "_ref", "pydeseq2")]
__version__ = "0.5.3"
