"""List files for the drop-in programs (TEST INFRASTRUCTURE).

The programs read every entry of a list file as a token of at most 99 characters (fscanf("%s") into char[100], as the
reference does; tests/test_host_cpu.py::test_read_list_tokens pins it), and the trainer cuts its report's name from the
first 99 characters of its output path (T-FS:205-207).  An absolute path under a deep temporary directory can be longer,
so the tests run the programs from their temporary directory and name the files relative to it.
"""
import os


def write_list(path, entries):
    """Writes a list file with one entry per line, each relative to the list's own directory (which the caller makes the
    working directory of the program that reads it)."""
    d = os.path.dirname(str(path))
    with open(path, "w") as f:
        f.write("".join(os.path.relpath(str(e), d) + "\n" for e in entries))
