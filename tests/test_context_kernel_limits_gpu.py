"""Several render contexts in one process share each kernel's opt-in shared-memory limit (it belongs to the kernel, not to
a context).  A context that first launches the primary kernel with little shared memory must not leave the limit below
what another context has already launched it with: that context's next frame of the same scene would fail with
'invalid argument'."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_a_new_context_does_not_lower_the_limit_of_an_older_one(pkg):
    pkg.build.build_library()
    big = pkg.scene.reference_scene(1024, 1)     # sphere records resident: about 18 KB of dynamic shared memory
    small = pkg.scene.reference_scene(1, 9)      # about 1 KB
    cam = pkg.scene.reference_camera()
    a = pkg.Renderer(0)
    b = pkg.Renderer(0)
    try:
        a.set_scene(big)
        first = a.render(cam, 96, 54).copy()
        b.set_scene(small)
        b.render(cam, 96, 54)
        again = a.render(cam, 96, 54)
        assert np.array_equal(first, again)
        # and the other way round: the small context keeps rendering after the big one's launches
        assert np.array_equal(b.render(cam, 96, 54), b.render(cam, 96, 54))
    finally:
        b.close()
        a.close()
