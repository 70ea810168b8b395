"""Test doubles for the control plane either side of the path: a stateful mock kube-apiserver +
kubelet /pods/ endpoint, a fake kubelet Registration server, and synthetic cluster generators for
SURVEY.md §8(d) configs 4-5. Used by tests/ and by bench_allocate; never by the plugin itself."""
import tempfile


def socket_dir(prefix: str) -> str:
    """A fresh directory for unix sockets. A socket's path may not exceed 107 bytes, so where the temporary
    directory is a deep one (a long TMPDIR) it is made under /tmp instead."""
    root = tempfile.gettempdir()
    return tempfile.mkdtemp(prefix=prefix, dir=root if len(root) <= 40 else "/tmp")
