"""Stand-in for the reference's robot demo (robot-visualization.py), with the process layout scripts/run_demo.py has
to handle: the UI process imports ``from gicp import gicp, apply_transformation`` and runs a 10 fps loop in which a
robot scans a 2-D world with a ray caster; every pair of consecutive scans goes to a GICP worker in a FORKED process
through queues (lists of tuples in, the pickled result out, each call padded to 0.5 s), and the UI integrates the
returned transforms into a pose estimate.  The script ends with sys.exit()."""
import math
import multiprocessing
import sys
import time

import numpy as np
import pygame
from gicp import apply_transformation, gicp

NUM_RAYS, MAX_RANGE, SPEED, YAW_SPEED, NOISE = 90, 400, 2, 2, 2
OBSTACLES = [pygame.Rect(100, 250, 200, 50), pygame.Rect(400, 450, 50, 200), (600, 300, 50), (200, 550, 75)]


def ray_segment(p1, p2, p3, p4):
    (x1, y1), (x2, y2), (x3, y3), (x4, y4) = p1, p2, p3, p4
    denom = (x1 - x2) * (y3 - y4) - (y1 - y2) * (x3 - x4)
    if denom == 0:
        return None
    t = ((x1 - x3) * (y3 - y4) - (y1 - y3) * (x3 - x4)) / denom
    u = -((x1 - x2) * (y1 - y3) - (y1 - y2) * (x1 - x3)) / denom
    return (x1 + t * (x2 - x1), y1 + t * (y2 - y1)) if 0 <= t <= 1 and 0 <= u <= 1 else None


def ray_circle(p1, p2, center, radius):
    dx, dy = p2[0] - p1[0], p2[1] - p1[1]
    fx, fy = p1[0] - center[0], p1[1] - center[1]
    a, b, c = dx * dx + dy * dy, 2 * (fx * dx + fy * dy), fx * fx + fy * fy - radius * radius
    disc = b * b - 4 * a * c
    if disc < 0:
        return []
    ts = ((-b - math.sqrt(disc)) / (2 * a), (-b + math.sqrt(disc)) / (2 * a))
    return [(p1[0] + t * dx, p1[1] + t * dy) for t in ts if 0 <= t <= 1]


def cast_ray(x, y, angle):
    end = (x + MAX_RANGE * math.cos(math.radians(angle)), y + MAX_RANGE * math.sin(math.radians(angle)))
    hits = []
    for ob in OBSTACLES:
        if isinstance(ob, pygame.Rect):
            for a, b in ((ob.topleft, ob.topright), (ob.topright, ob.bottomright),
                         (ob.bottomright, ob.bottomleft), (ob.bottomleft, ob.topleft)):
                p = ray_segment((x, y), end, a, b)
                if p:
                    hits.append(p)
        else:
            hits += ray_circle((x, y), end, ob[:2], ob[2])
    if not hits:
        return None
    return min(math.hypot(p[0] - x, p[1] - y) for p in hits) + np.random.uniform(-NOISE, NOISE)


def scan(x, y, yaw):
    """Robot-relative hit points as a list of tuples."""
    points = []
    for angle in range(yaw, yaw + 360, 360 // NUM_RAYS):
        d = cast_ray(x, y, angle)
        if d:
            points.append((d * math.cos(math.radians(angle - yaw)), d * math.sin(math.radians(angle - yaw))))
    return points


def gicp_worker(requests, results):
    while True:
        job = requests.get()
        if job is None:
            return
        start = time.time()
        results.put(gicp(job[0], job[1], max_distance_nearest_neighbors=200, tolerance=1))
        time.sleep(max(0.0, 0.5 - (time.time() - start)))


def main():
    pygame.init()
    screen = pygame.display.set_mode((800, 700))
    clock = pygame.time.Clock()
    ctx = multiprocessing.get_context("fork")
    requests, results = ctx.Queue(), ctx.Queue()
    worker = ctx.Process(target=gicp_worker, args=(requests, results), daemon=True)
    worker.start()

    x, y, yaw = 50.0, 400.0, 0
    estimate = [x, y, 0.0]
    previous, busy, running = None, False, True
    while running:
        for event in pygame.event.get():
            if event.type == pygame.QUIT:
                running = False
        keys = pygame.key.get_pressed()
        yaw += YAW_SPEED * (keys[pygame.K_RIGHT] - keys[pygame.K_LEFT])
        step = SPEED * (keys[pygame.K_UP] - keys[pygame.K_DOWN])
        x, y = x + step * math.cos(math.radians(yaw)), y + step * math.sin(math.radians(yaw))
        current = scan(x, y, yaw)
        if busy and not results.empty():
            T = results.get()[0]
            busy = False
            c, s = math.cos(math.radians(estimate[2])), math.sin(math.radians(estimate[2]))
            estimate[0] -= c * T[0, 2] - s * T[1, 2]
            estimate[1] -= s * T[0, 2] + c * T[1, 2]
            estimate[2] -= math.degrees(math.atan2(T[1, 0], T[0, 0]))
        if not busy:
            if previous is not None:
                requests.put((previous, current))
                busy = True
            previous = current

        screen.fill((0, 0, 0))
        c, s = math.cos(math.radians(yaw)), math.sin(math.radians(yaw))
        pose = np.array([[c, -s, x], [s, c, y], [0.0, 0.0, 1.0]])
        for p in apply_transformation(np.asarray(current).reshape(-1, 2), pose):
            pygame.draw.circle(screen, (0, 255, 0), (int(p[0]), int(p[1])), 2)
        pygame.draw.circle(screen, (255, 0, 0), (int(estimate[0]), int(estimate[1])), 5)
        pygame.display.flip()
        clock.tick(10)

    requests.put(None)
    if busy:
        results.get()          # the answer still in flight: the worker exits once its queue is drained
    worker.join()
    pygame.quit()
    sys.exit()


if __name__ == "__main__":
    main()
