"""Stand-in for the reference's static viewer (visualization.py), with the structure scripts/run_demo.py has to
handle: ``from gicp import gicp, apply_transformation`` resolved by whoever runs the script, one gicp() call on the
circle + square pair of BASELINE config 1, then a pygame loop that steps through the iterations on the arrow keys
until QUIT.  With random / numpy.random seeded to s, the pair is tests/demo_inputs.config1_pair(s)."""
import random

import numpy as np
import pygame
from gicp import apply_transformation, gicp


def square_points(center, size, per_side):
    half = size / 2
    xs = np.linspace(center[0] - half, center[0] + half, per_side)
    ys = np.linspace(center[1] - half, center[1] + half, per_side)
    pts = [[x, center[1] - half] for x in xs] + [[center[0] + half, y] for y in ys]
    pts += [[x, center[1] + half] for x in xs] + [[center[0] - half, y] for y in ys]
    keep = random.sample(range(len(pts)), len(pts) // 2)
    return np.array([pts[i] for i in range(len(pts)) if i in keep])


def circle_points(center, radius, count):
    angles = [random.uniform(0, 2 * np.pi) for _ in range(count)]
    return np.array([[center[0] + radius * np.cos(a), center[1] + radius * np.sin(a)] for a in angles])


def main():
    source = np.concatenate([circle_points((300, 150), 100, 30), square_points((600, 250), 200, 30)])
    ang = np.pi / 3
    rot = np.array([[np.cos(ang), -np.sin(ang)], [np.sin(ang), np.cos(ang)]])
    target = np.dot(source, rot.T) + np.array([150, -50])
    source = source + np.random.normal(0, 2, source.shape)
    target = target + np.random.normal(0, 5, target.shape)
    np.random.shuffle(target)
    target = target[:len(target) - 3]

    T, all_T, source_cov, target_cov, hw_source, hw_target, all_source_cov = gicp(source, target)

    pygame.init()
    screen = pygame.display.set_mode((1000, 700))
    pygame.display.set_caption("GICP iterations")
    clock = pygame.time.Clock()
    step, running = 0, True
    while running:
        for event in pygame.event.get():
            if event.type == pygame.QUIT:
                running = False
            elif event.type == pygame.KEYDOWN and event.key == pygame.K_RIGHT:
                step = min(step + 1, len(all_T) - 1)
            elif event.type == pygame.KEYDOWN and event.key == pygame.K_LEFT:
                step = max(step - 1, 0)
        screen.fill((255, 255, 255))
        for p in target:
            pygame.draw.circle(screen, (0, 0, 255), (int(p[0]), int(p[1])), 3)
        for p in apply_transformation(source, all_T[step]):
            pygame.draw.circle(screen, (255, 0, 0), (int(p[0]), int(p[1])), 3)
        pygame.display.flip()
        clock.tick(30)
    pygame.quit()


if __name__ == "__main__":
    main()
